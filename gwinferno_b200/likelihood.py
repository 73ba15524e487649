"""Reference-facing front-end of the fused population likelihood.

:func:`hierarchical_likelihood` keeps the signature of the reference's
``gwinferno.pipeline.analysis.hierarchical_likelihood`` (analysis.py:139-163) but takes the LAZY
weights produced by the mirror model classes (gwinferno_b200/models.py) and evaluates the whole
path -- per-sample densities, per-event and injection Monte-Carlo sums, N_eff / variance cuts and
the gradient with respect to every hyper-parameter -- in one call into libgwi.so.  Without
NumPyro in the loop the "sites" the reference records with ``numpyro.deterministic`` /
``numpyro.factor`` (analysis.py:260-319) are returned in a :class:`LikelihoodResult`.

There is no CPU fallback: a missing library or GPU raises :class:`gwinferno_b200.capi.GwiError`.
"""

import collections
import os
import warnings

import numpy as np

from . import capi, lowering

# device-resident plans, keyed by the uids of the model objects / sample arrays of a weight product
# (models._uid_of: never re-used, unlike id()); least-recently-used plans are closed when more than
# GWI_MAX_ENGINES (default 8) are alive -- a cfg-3 plan is 7.4 GB of device memory
_ENGINES = collections.OrderedDict()
_MAX_ENGINES = max(1, int(os.environ.get("GWI_MAX_ENGINES", "8")))
_BUILDS = collections.Counter()  # (term kinds, sharing pattern) -> plans built; warns when one model shape keeps missing the cache


class PopulationLikelihood:
    """Device-resident plan for one (catalog, population model) pair; evaluate for many Lambda."""

    def __init__(self, lowered, total_inj, device=0, need_neff_grad=False, chunk_steps=0, n_deep=-1, batch_hint=0, catalog_on_device=False,
                 keep_sample_index=False):
        """keep_sample_index=True: the device plan also records each sample's catalog position (4 bytes per sample), which
        :meth:`sample_log_weights` and :meth:`posterior_predictive` need."""
        self.lowered = lowered
        self.spec = lowered.spec
        self.n_params = lowered.spec.n_params
        # catalog_on_device=True: the sample columns are placed in device memory first and the plan is built from there
        # (capi.Catalog(on_device=True)): the setting of a caller whose arrays already live on the GPU
        self.catalog = capi.Catalog(lowered.pe_cols, lowered.inj_cols, total_inj, device=device, on_device=catalog_on_device)
        self.model = capi.Model(self.catalog, lowered.spec, need_neff_grad=need_neff_grad, chunk_steps=chunk_steps, n_deep=n_deep, batch_hint=batch_hint,
                                keep_sample_index=keep_sample_index)
        self.need_neff_grad = need_neff_grad
        self.n_events = self.catalog.n_events

    @classmethod
    def from_weights(cls, pe_weights, inj_weights, total_inj, **kw):
        return cls(lowering.lower(pe_weights, inj_weights), total_inj, **kw)

    def evaluate(self, lam, jacobians=True):
        """``logBF[E], logNeff[E], log_mu, logNeff_inj`` (+ Jacobians) -- the outputs of the
        reference's per_event_log_bayes_factors / detection_efficiency (analysis.py:50-136)."""
        return self.model.evaluate(lam, jacobians=jacobians)

    def loglike(self, lam, Nobs=None, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False):
        """``(log_l, dlog_l/dLambda, diagnostics)`` through gwi_loglike_host (host buffers)."""
        if marginalize_selection and not self.need_neff_grad:
            raise ValueError("marginalize_selection=True needs PopulationLikelihood(..., need_neff_grad=True)")
        head, grad = self.model.loglike_host(
            lam, self.n_events if Nobs is None else Nobs, marginalize_selection=marginalize_selection, min_neff_cut=min_neff_cut, max_variance_cut=max_variance_cut
        )
        return head["log_l"], grad, head

    def last_sites(self):
        """Per-event sites of the LAST evaluation (analysis.py:260-264): ``logBFs``, ``log_nEffs``,
        ``variance_log_BFs`` [E] and ``variance_log_detection_efficiency``, read back from the device."""
        seg = self.model.last_sites()
        return {"logBFs": seg[1:, 0].copy(), "log_nEffs": seg[1:, 1].copy(), "variance_log_BFs": seg[1:, 2].copy(), "variance_log_detection_efficiency": float(seg[0, 2])}

    def info(self):
        return self.model.info()

    def sample_log_weights(self, lam, host_log_norm=0.0):
        """Per-sample population log-weights ``log p_pop(theta | Lambda) - log prior(theta)``, every normaliser included
        (``-inf`` where the weight is 0): ``(pe, inj)`` with ``pe`` ``(E, S)`` (a list of per-event arrays for ragged
        events) and ``inj`` ``(I,)``.  ``host_log_norm``: the host-side normaliser of the weights
        (``lowering.host_log_norm(pe_weights, n_params)[0]``), subtracted here, so that ``logsumexp(pe[i]) - log S_i`` is
        the ``logBFs`` site of event i and ``logsumexp(inj) - log total_inj`` the log detection efficiency.  Exponentiated
        and normalised per event they are the population-reweighted event posteriors."""
        x = self.model.sample_log_weights(lam) - float(host_log_norm)
        off = self.catalog.offsets
        pe = [x[off[i] : off[i + 1]] for i in range(self.n_events)]
        if self.n_events and len({a.size for a in pe}) == 1:
            pe = x[: off[-1]].reshape(self.n_events, -1)
        return pe, x[off[-1] :]

    def posterior_predictive(self, lam, seed=0, draws_per_event=1, draws_inj=None):
        """Weighted draws (the reference's posterior-predictive resampling, analysis.py:321-355): ``(pe_idx[E,
        draws_per_event], inj_idx[draws_inj])`` int64 sample indices inside each event / into the injection columns, drawn
        with probability proportional to the weight; -1 where an event (or the injection set) has no weight.
        ``draws_inj`` defaults to E.  Counter-based (Philox4x32-10 keyed by ``seed``): the same arguments give the same
        draws, whatever the plan geometry."""
        return self.model.draw_samples(lam, seed, draws_per_event, self.n_events if draws_inj is None else draws_inj)


class LikelihoodResult:
    """What the reference's hierarchical_likelihood leaves in the NumPyro trace (analysis.py:260-319)."""

    def __init__(self, log_l, grad_flat, head, lowered, pe_weights, surveyed_hypervolume, Tobs, Nobs):
        self.log_likelihood = float(log_l)
        self.grad_flat = grad_flat
        self.sites = {
            "log_l": float(log_l),
            "log_nEff_inj": head["logNeff_inj"],
            "detection_efficiency": float(np.exp(head["log_mu"])),
            "sum_logBFs": head["sum_logBF"],
            "variance_log_likelihood": head["variance"],
            "passed_cuts": bool(head["passed"]),
        }
        # per-event sites of analysis.py:260-264 (read back from the device results of this evaluation)
        for k in ("logBFs", "log_nEffs", "variance_log_BFs", "variance_log_detection_efficiency"):
            if k in head:
                self.sites[k] = head[k]
        if surveyed_hypervolume is not None:
            self.sites["surveyed_hypervolume"] = float(surveyed_hypervolume) / 1.0e9 * Tobs
        self._lowered = lowered
        self._pe_weights = pe_weights
        self.rate = None
        self.ppc = None  # posterior_predictive_check=True: {"obs_index", "pred_index", "obs": {name: [E]}, "pred": {name: [E]}}

    def grad(self, param):
        """Gradient of log_l with respect to a parameter OBJECT that was passed to the model calls
        (the total derivative: summed over every argument position the object was passed to)."""
        if self._lowered is None:  # cached engine: the object -> Lambda slots map of THIS call's parameter objects
            e = self._engine_lowered
            self._lowered = lowering.Lowered(e.spec, e.pe_cols, e.inj_cols, e.param_layout, lowering.object_slot_map(self._pe_weights))
        sl = self._lowered.all_slots_for(param)
        g = self.grad_flat[sl[0]]
        for extra in sl[1:]:
            g = g + self.grad_flat[extra]
        return g


def hierarchical_likelihood(
    pe_weights,
    inj_weights,
    total_inj,
    Nobs,
    Tobs,
    surveyed_hypervolume=None,
    categorical=False,
    marginal_qs=False,
    indv_weights=None,
    rngkey=None,
    pop_frac=None,
    reconstruct_rate=True,
    marginalize_selection=False,
    min_neff_cut=True,
    max_variance_cut=False,
    posterior_predictive_check=False,
    param_names=None,
    pedata=None,
    injdata=None,
    m2min=3.0,
    m1min=5.0,
    mmax=100.0,
    log=False,
    device=0,
):
    """Drop-in for ``gwinferno.pipeline.analysis.hierarchical_likelihood`` (analysis.py:139-356)
    on lazy weights.  ``log=True`` takes lazy LOG-weights (``log_prob`` terms combined with ``+`` and
    ``- jnp.log(prior)``, analysis.py:401-421); the fused path always works in log space, so both forms
    lower to the same device model.  The categorical sub-population branch (:246-254) is outside the fused path
    and raises NotImplementedError.

    ``posterior_predictive_check=True`` (:321-355) needs ``param_names``, ``pedata`` (dict name -> ``(E, S)`` array, or a
    list of per-event arrays) and ``injdata`` (dict name -> ``(I,)`` array); without them it raises NotImplementedError.
    It evaluates on a device plan that keeps each sample's catalog position (a separate cached engine) and draws, with
    probability proportional to the population weight, one PE sample per event and E found injections on the GPU
    (``PopulationLikelihood.posterior_predictive``, Philox4x32-10 keyed by ``rngkey``, 0 when None; not JAX's stream).
    The drawn values are returned in ``res.ppc = {"obs_index", "pred_index", "obs": {name: [E]}, "pred": {name: [E]}}``
    and as the sites ``{name}_obs_event_{i}`` / ``{name}_pred_event_{i}`` (NaN where an event has no weight); ``log_l``
    and the gradient are those of the call without it.  The reference's source was not available when this was
    written: these site names follow its description, not its code, and ``m1min`` / ``m2min`` / ``mmax``, whose role
    there could not be checked, are accepted and unused.

    ``reconstruct_rate`` (:265-268): NumPyro
    draws ``unscaled_rate ~ Gamma(Nobs)`` from the trace's key; here it is drawn from
    ``numpy.random.default_rng(rngkey)`` (``rngkey``: an int seed or ``None``) when a surveyed hypervolume is
    given, and returned -- as in the reference -- as the function's ``rate`` (``LikelihoodResult.rate``)."""
    if max_variance_cut and (marginalize_selection or min_neff_cut):
        raise ValueError(
            "max_variance_cut is True which requires marginalize_selection and min_neff_cut to be False but got "
            f"marginalize_selection = {marginalize_selection} and min_neff_cut = {min_neff_cut}"
        )
    if bool(log) != bool(getattr(pe_weights, "log_domain", False)) or bool(log) != bool(getattr(inj_weights, "log_domain", False)):
        raise ValueError("log=True expects log-weights (built from log_prob with + / -), log=False expects weights (built with * and /)")
    if categorical or marginal_qs:
        raise NotImplementedError("the categorical sub-population branch is not part of the fused path")
    ppc = bool(posterior_predictive_check)
    if ppc and (param_names is None or pedata is None or injdata is None):
        raise NotImplementedError("posterior_predictive_check=True needs param_names, pedata and injdata (the sample values the draws are read from)")
    keys, pattern = lowering._structure(pe_weights, inj_weights)
    cache_key = (keys, pattern, float(total_inj), bool(marginalize_selection), int(device), ppc)
    eng = _ENGINES.get(cache_key)
    if eng is None:
        shape_key = (tuple(k[0] if isinstance(k[0], str) else k[1] for k in keys), pattern)
        _BUILDS[shape_key] += 1
        if _BUILDS[shape_key] == 4:
            warnings.warn("hierarchical_likelihood built a new device plan for the same model shape 4 times: a model object or sample array is "
                          "re-created on every call (construct the models once, outside the sampled function)", RuntimeWarning, stacklevel=2)
        extra = dict(keep_sample_index=True) if ppc else {}
        eng = PopulationLikelihood.from_weights(pe_weights, inj_weights, total_inj, device=device, need_neff_grad=bool(marginalize_selection), **extra)
        _ENGINES[cache_key] = eng
        while len(_ENGINES) > _MAX_ENGINES:
            _, old = _ENGINES.popitem(last=False)
            old.model.close()
            old.catalog.close()
        lowered = eng.lowered
    else:
        _ENGINES.move_to_end(cache_key)
        # same static structure, new hyper-parameter objects: the slot map is rebuilt on demand (LikelihoodResult.grad)
        lowered = None
    lam = lowering.flatten_params(pe_weights, eng.n_params)
    log_l, grad, head = eng.loglike(lam, Nobs=Nobs, marginalize_selection=marginalize_selection, min_neff_cut=min_neff_cut, max_variance_cut=max_variance_cut)
    head = dict(head)
    head.update(eng.last_sites())
    # O(P) host glue: chain rule through parameter maps; per-sample constants kept off the device
    grad = lowering.pull_back(pe_weights, grad)
    log_l, grad, head = apply_host_norm(log_l, grad, head, *lowering.host_log_norm(pe_weights, eng.n_params), n_events=eng.n_events, Nobs=Nobs)
    res = LikelihoodResult(log_l, grad, head, lowered, pe_weights, surveyed_hypervolume, Tobs, Nobs)
    res._engine_lowered = eng.lowered
    if reconstruct_rate and surveyed_hypervolume is not None:
        # analysis.py:265-268
        total_vt = float(surveyed_hypervolume) / 1.0e9 * Tobs
        unscaled = float(np.random.default_rng(rngkey).gamma(Nobs))
        res.sites["unscaled_rate"] = unscaled
        res.rate = res.sites["rate"] = unscaled / float(np.exp(head["log_mu"])) / total_vt
    if ppc:
        _posterior_predictive(res, eng, lam, rngkey, param_names, pedata, injdata)
    return res


def _seed_of(rngkey):
    """An integer seed from ``rngkey``: an int, None (0), or an array of key words (the last two, as JAX keys hold them)."""
    if rngkey is None:
        return 0
    w = np.asarray(rngkey).ravel()
    if w.size == 1:
        return int(w[0]) & 0xFFFFFFFFFFFFFFFF
    return ((int(w[-2]) & 0xFFFFFFFF) << 32) | (int(w[-1]) & 0xFFFFFFFF)


def _posterior_predictive(res, eng, lam, rngkey, param_names, pedata, injdata):
    """One PE sample per event ("obs") and E found injections ("pred") drawn by weight (analysis.py:321-355)."""
    E = eng.n_events
    pe_idx, inj_idx = eng.posterior_predictive(lam, seed=_seed_of(rngkey), draws_per_event=1, draws_inj=E)
    obs_index = pe_idx[:, 0]
    obs, pred = {}, {}
    for name in param_names:
        ev = pedata[name]
        obs[name] = np.array([np.asarray(ev[i], dtype=np.float64)[obs_index[i]] if obs_index[i] >= 0 else np.nan for i in range(E)])
        inj = np.asarray(injdata[name], dtype=np.float64)
        pred[name] = np.where(inj_idx >= 0, inj[np.maximum(inj_idx, 0)], np.nan) if inj.size else np.full(inj_idx.shape, np.nan)
        for i in range(E):
            res.sites[f"{name}_obs_event_{i}"] = float(obs[name][i])
            res.sites[f"{name}_pred_event_{i}"] = float(pred[name][i])
    res.ppc = {"obs_index": obs_index, "pred_index": inj_idx, "obs": obs, "pred": pred}


def apply_host_norm(log_l, grad, head, logZ, dlogZ, n_events, Nobs):
    """Every sample weight is ``exp(-logZ)`` times what the device model evaluated: shift the sites
    (``logBF_i`` and ``log mu`` by ``-logZ``; N_eff and the variances are scale-free) and the
    likelihood ``log_l = sum_i logBF_i - Nobs log mu`` (analysis.py:257-319) by ``(Nobs - E) logZ``
    -- nothing when ``Nobs`` equals the number of events, as in every reference example."""
    if logZ == 0.0 and not np.any(dlogZ):
        return log_l, grad, head
    head = dict(head)
    head["log_mu"] = head["log_mu"] - logZ
    head["sum_logBF"] = head["sum_logBF"] - n_events * logZ
    if "logBFs" in head:
        head["logBFs"] = head["logBFs"] - logZ
    if head["passed"]:
        log_l = log_l + (Nobs - n_events) * logZ
        grad = grad + (Nobs - n_events) * dlogZ
    return log_l, grad, head


def clear_cache():
    for e in _ENGINES.values():
        e.model.close()
        e.catalog.close()
    _ENGINES.clear()
