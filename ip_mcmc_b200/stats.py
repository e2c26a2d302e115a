"""Chain statistics: the reference's autocorrelation (sampler.py:43-54, helpers.py:41-54,
utilities.py:169-186) and the ESS estimator SURVEY.md section 8(d) defines on top of it.
Host-side NumPy by design (SURVEY.md section 8(a) row T1): it post-processes recorded traces."""
import numpy as np


def autocorr(x):
    """Lag-0-normalised biased autocorrelation (MCMCSampler.autocorr, sampler.py:43-54);
    a constant series gives all ones."""
    x = np.asarray(x, dtype=np.float64)
    x_ = x - np.mean(x)
    n = x_.shape[0]
    # np.correlate(x_, x_, 'full')[-n:] via FFT for long chains (same values to rounding)
    if n > 2048:
        m = 1 << int(np.ceil(np.log2(2 * n)))
        f = np.fft.rfft(x_, m)
        result = np.fft.irfft(f * np.conj(f), m)[:n]
    else:
        result = np.correlate(x_, x_, mode="full")[-n:]
    if result[0] == 0:
        return np.ones_like(result)
    return result / result[0]


def windowed_autocorrelation(samples, tau_max):
    """helpers.autocorrelation (helpers.py:41-54): samples [n_vars, n]; average of autocorr over
    consecutive windows of length tau_max."""
    samples = np.asarray(samples)
    avg_over = int(samples.shape[1] / tau_max)
    assert avg_over > 0, "Not enough samples to compute autocorrelation with specified length"
    ac = np.zeros((samples.shape[0], tau_max))
    for i in range(avg_over):
        for var in range(samples.shape[0]):
            ac[var] += autocorr(samples[var, i * tau_max:(i + 1) * tau_max])
    return ac / avg_over


def uncorrelated_sample_spacing(x, threshold=1e-3):
    """tau_0 of the reference (report/scripts/burgers/utilities.py:169-186), restated faithfully:
    x [n_vars, n]; the window length tau starts at 10 and grows by x1.5 (truncated) per round; each round
    averages the windowed autocorrelation (helpers.py:41-54) over the variables and returns the first lag
    at which it is <= 0.001.  When fewer than two windows of the current tau fit into the chain the
    reference gives up and returns ``len(x)`` -- the number of VARIABLES, since x is [n_vars, n] (kept)."""
    x = np.asarray(x)
    tau = 10
    while True:
        if 2 > int(len(x[0, :]) / tau):
            return len(x)              # "never decorrelate"
        tau = int(tau * 1.5)
        avg_ac = np.mean(windowed_autocorrelation(x, tau), axis=0)
        idx = np.argwhere(avg_ac <= threshold)
        if len(idx) > 0:
            return int(idx[0][0])


def fixed_window_sample_spacing(samples, tau_max=100, threshold=1e-3):
    """First lag at which the variable-averaged windowed autocorrelation of ONE window length tau_max
    drops to <= threshold (tau_max if it never does).  Not the reference's definition (see
    uncorrelated_sample_spacing): a fixed window makes sweep points comparable."""
    ac = np.mean(windowed_autocorrelation(samples, tau_max), axis=0)
    below = np.nonzero(ac <= threshold)[0]
    return int(below[0]) if below.size else int(tau_max)


def integrated_autocorr_time(x):
    """tau = 1 + 2 * sum_k rho_k with Geyer's initial-positive-sequence cut-off (pairs
    rho_{2m} + rho_{2m+1} summed while positive)."""
    rho = autocorr(x)
    n = rho.shape[0]
    tau = 1.0
    k = 1
    while k + 1 < n:
        pair = rho[k] + rho[k + 1]
        if pair <= 0:
            break
        tau += 2.0 * pair
        k += 2
    return max(tau, 1.0)


def ess(samples):
    """samples [n, d] of ONE chain -> per-parameter ESS = n / tau."""
    samples = np.asarray(samples, dtype=np.float64)
    n = samples.shape[0]
    return np.array([n / integrated_autocorr_time(samples[:, j]) for j in range(samples.shape[1])])


def ess_multichain(traces):
    """traces [n_chains, n, d] -> (total ESS = sum over chains of min over parameters, per-chain)."""
    per = np.array([ess(t).min() for t in traces])
    return float(per.sum()), per


def split_sequences(traces):
    """traces [M, n, d] -> the 2M split sequences [2M, h, d], h = n // 2: the first and the last h draws of
    each chain (the middle draw of an odd n is dropped), sequence 2c and 2c+1 from chain c."""
    x = np.asarray(traces, dtype=np.float64)
    if x.ndim != 3 or x.shape[1] < 4:
        raise ValueError("traces must be [n_chains, n >= 4, d], got %s" % (x.shape,))
    h = x.shape[1] // 2
    return np.stack([x[:, :h], x[:, x.shape[1] - h:]], axis=1).reshape(-1, h, x.shape[2])


def _split_var_plus(psi):
    """(W, var+) of split sequences psi [m, h, d] (BDA3 section 11.4)."""
    m, h = psi.shape[0], psi.shape[1]
    means = psi.mean(axis=1)
    W = psi.var(axis=1, ddof=1).mean(axis=0)
    B = h / (m - 1) * ((means - means.mean(axis=0)) ** 2).sum(axis=0)
    return W, (h - 1) / h * W + B / h


def split_rhat(traces):
    """Split-R-hat (BDA3 section 11.4) of traces [M, n, d] -> [d]: sqrt(var+ / W) over the 2M half-chains.
    All sequences constant gives NaN (0/0), constant sequences at different values inf."""
    with np.errstate(divide="ignore", invalid="ignore"):
        W, var_plus = _split_var_plus(split_sequences(traces))
        return np.sqrt(var_plus / W)


def multichain_ess(traces):
    """Multi-chain effective sample size (BDA3 section 11.5, variogram form) of traces [M, n, d] on the split
    sequences -> (n_eff [d], T [d]).  rho_t = 1 - V_t / (2 var+), V_t the mean squared difference of draws t
    apart; the sum of rho_t runs over t = 1, 2, ... and stops at the first odd T with
    rho_{T+1} + rho_{T+2} < 0 (or T + 2 > h - 1); n_eff = m h / (1 + 2 S)."""
    psi = split_sequences(traces)
    m, h, d = psi.shape
    n_eff, cutoff = np.empty(d), np.empty(d, dtype=np.int64)
    with np.errstate(divide="ignore", invalid="ignore"):
        _, var_plus = _split_var_plus(psi)
        for j in range(d):
            def rho(t):
                V = ((psi[:, t:, j] - psi[:, :h - t, j]) ** 2).sum() / (m * (h - t))
                return 1.0 - V / (2.0 * var_plus[j])
            S, t = 0.0, 1
            while True:
                S += rho(t)
                if t + 2 > h - 1 or rho(t + 1) + rho(t + 2) < 0:
                    break
                S += rho(t + 1)
                t += 2
            n_eff[j], cutoff[j] = m * h / (1.0 + 2.0 * S), t
    return n_eff, cutoff


def usable_samples(n, burn_in, tau0):
    """M = (N - b) / tau_0 (report/burgers.org:43-45)."""
    return (n - burn_in) / max(tau0, 1)


def merge_moments(parts):
    """Chan et al. merge of (n, mean[d], M2[d]) triples -> (n, mean, M2)."""
    n, mean, m2 = 0.0, None, None
    for nb, mb, Mb in parts:
        if nb <= 0:
            continue
        mb, Mb = np.asarray(mb, dtype=np.float64), np.asarray(Mb, dtype=np.float64)
        if mean is None:
            n, mean, m2 = float(nb), mb.copy(), Mb.copy()
            continue
        nt = n + nb
        delta = mb - mean
        mean = mean + delta * (nb / nt)
        m2 = m2 + Mb + delta * delta * (n * nb / nt)
        n = nt
    return n, mean, m2
