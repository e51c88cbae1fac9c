"""float64 numpy oracle of the ensemble scores (cesm_ensemble_scores), from the direct O(n^2) definitions."""
import numpy as np


def ensemble_scores(pred, target, chunk_elems=1 << 24):
    """pred [T, n, HW], target [T, m, HW] -> dict of float64 [T, HW] maps and the int64 [T, n+1] rank histogram,
    with the kernel's rules: fair CRPS (Ferro 2014) averaged over the targets, bias, ddof-1 spreads, ensemble-mean MSE;
    bin r = #{i : x_i < y_j} (a tie is not below); a column holding a non-finite value is NaN in every map and left
    out of the histogram."""
    x = np.asarray(pred, np.float64)
    y = np.asarray(target, np.float64)
    T, n, HW = x.shape
    m = y.shape[1]
    maps = {k: np.empty((T, HW)) for k in ("crps", "bias", "sd_pred", "sd_target", "mse_mean")}
    hist = np.zeros((T, n + 1), np.int64)
    iu, ku = np.triu_indices(n, 1)
    step = max(1, chunk_elems // (T * n * max(n, m)))  # pixels per chunk: bounds the pairwise temporaries
    for p0 in range(0, HW, step):
        xs, ys = x[:, :, p0:p0 + step], y[:, :, p0:p0 + step]
        bad = ~(np.isfinite(xs).all(1) & np.isfinite(ys).all(1))                  # [T, P]
        xy = np.abs(xs[:, :, None, :] - ys[:, None, :, :]).mean(axis=(1, 2))      # mean_j (1/n) sum_i |x_i - y_j|
        xx = np.abs(xs[:, iu, :] - xs[:, ku, :]).sum(1) / (n * (n - 1))            # 1/(n(n-1)) sum_{i<k} |x_i - x_k|
        mx = xs.mean(1)
        part = {"crps": xy - xx, "bias": mx - ys.mean(1), "sd_pred": xs.std(1, ddof=1),
                "sd_target": ys.std(1, ddof=1), "mse_mean": ((mx[:, None, :] - ys) ** 2).mean(1)}
        for k, v in part.items():
            v[bad] = np.nan
            maps[k][:, p0:p0 + step] = v
        ranks = (xs[:, :, None, :] < ys[:, None, :, :]).sum(1)                    # [T, m, P]
        for t in range(T):
            hist[t] += np.bincount(ranks[t][:, ~bad[t]].ravel(), minlength=n + 1)
    return {**maps, "rank_hist": hist}

def gaussian_crps(mu, sigma, y):
    """Closed-form CRPS of the forecast N(mu, sigma^2) at observation y: sigma [z (2 Phi(z) - 1) + 2 phi(z) - 1/sqrt(pi)]."""
    from scipy.stats import norm
    z = (np.asarray(y, np.float64) - mu) / sigma
    return sigma * (z * (2 * norm.cdf(z) - 1) + 2 * norm.pdf(z) - 1 / np.sqrt(np.pi))
