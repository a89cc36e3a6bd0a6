"""Reference evaluation of a double-lined binary for the tests, composed from the oracle's single-star pieces.

``binary_lnlike_batch`` calls ``oracle.payne_oracle.getspec`` once per component, with ``inst_R`` and ``outwave`` shared
and no polynomial, then forms m = (a_1 + k a_2) / (1 + k) with the blackbody flux ratio
k = Rratio^2 expm1(c2 / (lambda Teff_1)) / expm1(c2 / (lambda Teff_2)), multiplies by ``polycalc`` and takes chi2 in
float64 (include/payne_b200.h, PayneBinary).  No new numerics: at Rratio = 0 it is the single-star oracle.
"""
import numpy as np

from oracle import payne_oracle as O

C2_RAD = 1.438776877e8          # second radiation constant hc / k_B, AA K


def binary_lnlike_batch(cfg, theta, return_model=False, ideal_mlp=False):
    """``cfg`` as ``OracleLikelihood`` takes it.  The secondary's parameter P is ``P_sec`` of ``cfg.fitpars_i`` /
    ``cfg.fixedpars``, else the primary's; ``Rratio`` comes from the same place.  Returns lnL [B] (and the model
    [B, n_obs] and the components [B, 2, n_obs] with ``return_model``)."""
    net = O.make_net(cfg.spec, ideal=ideal_mlp)
    theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
    fit, fixed = list(cfg.fitpars_i), dict(cfg.fixedpars)
    w = np.asarray(cfg.obs_wave, dtype=np.float64)
    B = theta.shape[0]
    lnl = np.empty(B)
    model = np.empty((B, len(w)))
    comp = np.empty((B, 2, len(w)))
    for i in range(B):
        pd = {p: float(v) for p, v in zip(fit, theta[i])}
        pd.update(fixed)
        prim = {p: pd.get(p, np.nan) for p in O.SPEC_NAMES}
        sec = {p: pd.get(p + '_sec', prim[p]) for p in O.SPEC_NAMES}
        inst = O.FWHM_FACTOR_FIT * float(prim['Inst_R'])
        a = []
        for P in (prim, sec):
            _, f = O.getspec(net, cfg.spec, P['Teff'], P['log(g)'], P['[Fe/H]'], P['[a/Fe]'], P['Vmic'], P['Vrot'],
                             P['Vrad'], inst, w)
            a.append(np.asarray(f, dtype=np.float64))
        rr = float(pd['Rratio'])
        k = rr ** 2 * np.expm1(C2_RAD / (w * prim['Teff'])) / np.expm1(C2_RAD / (w * sec['Teff']))
        m = (a[0] + k * a[1]) / (1.0 + k)
        if cfg.runbools[2]:
            m = m * O.polycalc(np.array([pd[p] for p in fit if 'pc' in p]), w)
        model[i], comp[i, 0], comp[i, 1] = m, a[0], a[1]
        lnl[i] = -0.5 * np.sum(((m - cfg.obs_flux) ** 2.0) / (cfg.obs_eflux ** 2.0))
    if return_model:
        return lnl, model, comp
    return lnl
