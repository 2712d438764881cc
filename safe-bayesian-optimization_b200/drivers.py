"""The reference's BO loops as callable drivers (SURVEY.md section 8f row 3).

The reference keeps its acquisition loops in experiment scripts: ``test/test_SafeOpt.py:135-186`` (single
SafeOpt run with plot frames), ``:188-253`` (repeated runs written to ``data/*.npz``) and
``test/test_GoOSE.py:142-190``.  These functions are those loops, statement for statement in the decision rules,
over the drop-in ``models.SafeOpt.BO`` / ``models.GoOSE.BO`` objects -- so every ``Minimizer()``, ``Expander()``,
``Target()`` ... inside them is one pass of the CUDA grid pipeline instead of a differential-evolution run.
Everything here is host control flow: no numerics of its own.

The result files are written with ``numpy.savez`` of plain NumPy arrays in the reference's layout
(``data['0'] = {'sampled_x', 'sampled_output', 'observed_x', 'observed_output'}``), readable by the reference's
``utils/utils_solve_Benoit.py:16-64`` (``data[key].item()[...]``) without jax.
"""
from __future__ import annotations

import time

import numpy as np


def safeopt_iteration(GP_m, require_lipschitz_ucb=False):
    """One acquisition decision of SafeOpt.

    test/test_SafeOpt.py:144-158: ``x_new = minimizer if std_minimizer > std_expander else expander``.
    ``require_lipschitz_ucb`` adds the multi-run script's extra guard (``:228-240``): the expander is taken only if
    some constraint's ucb at the expander is >= 0.
    Returns (x_new, info)."""
    t0 = time.perf_counter()
    minimizer, std_minimizer = GP_m.Minimizer()
    expander, std_expander = GP_m.Expander()
    dt = time.perf_counter() - t0
    take_minimizer = std_minimizer > std_expander
    if require_lipschitz_ucb and not take_minimizer:
        ok = np.all(np.isfinite(expander)) and any(GP_m.ucb(expander, j) >= 0. for j in range(1, GP_m.n_fun))
        take_minimizer = not ok
    x_new = minimizer if take_minimizer else expander
    if not np.all(np.isfinite(x_new)):            # the other candidate may still exist (empty minimiser or expander set)
        x_new = expander if take_minimizer else minimizer
    _require_point(x_new, "SafeOpt: the safe set is empty on the grid (no minimiser and no expander)")
    return np.asarray(x_new, dtype=np.float64), {
        "minimizer": np.asarray(minimizer), "std_minimizer": float(std_minimizer),
        "expander": np.asarray(expander), "std_expander": float(std_expander),
        "chose": "minimizer" if take_minimizer else "expander", "acquisition_seconds": dt}


class EmptySafeSet(RuntimeError):
    """No grid point satisfies the safety constraints: there is nothing safe to sample.  The reference's DE always
    returns SOME point inside the bounds (feasible or not); sampling a non-finite point would poison the
    normalisation and the Cholesky factor of every later iteration, so the drivers stop instead."""


def _require_point(x, msg):
    if not np.all(np.isfinite(np.asarray(x, dtype=np.float64))):
        raise EmptySafeSet(msg)


def goose_iteration(GP_m):
    """One acquisition decision of GoOSE (test/test_GoOSE.py:151-162).  Returns (x_new, info)."""
    t0 = time.perf_counter()
    x_safe_min, min_safe_lcb = GP_m.minimize_obj_lcb()
    x_target, target_lcb = GP_m.Target()
    if min_safe_lcb <= target_lcb:
        x_new = x_safe_min
        x_target = np.array([np.nan] * GP_m.nx_dim)
        chose = "safe_minimum"
    else:
        x_new = GP_m.explore_safeset(x_target)
        chose = "explore"
    dt = time.perf_counter() - t0
    _require_point(x_new, "GoOSE: the safe set is empty on the grid (no safe minimum and no reachable target)")
    return np.asarray(x_new, dtype=np.float64), {
        "x_safe_min": np.asarray(x_safe_min), "min_safe_lcb": float(min_safe_lcb), "x_target": np.asarray(x_target),
        "target_lcb": float(target_lcb), "chose": chose, "acquisition_seconds": dt}


def _check_append_mode(hypopt, fixed_model):
    if fixed_model and hypopt is not None:
        raise ValueError("fixed_model keeps the installed hyper-parameters: pass hypopt=None")


def _append(GP_m, x, y, hypopt, fixed_model):
    if fixed_model:
        GP_m.add_sample_fixed(x, y)
    elif hypopt is None:
        GP_m.add_sample(x, y)
    else:
        GP_m.add_sample(x, y, hypopt=hypopt)


def run_safeopt(GP_m, n_iteration=10, noise=0., stop_std=0.01, on_iteration=None, require_lipschitz_ucb=False,
                hypopt=None, fixed_model=False):
    """test/test_SafeOpt.py:135-186 without the plotting side effects (pass ``on_iteration(i, GP_m, x_new, y, info)``
    to draw frames, e.g. with utils_SafeOpt.create_data_for_plot + plot_safe_region_Benoit).
    ``hypopt`` (additive): keep these hyper-parameters instead of refitting in every ``add_sample``.
    ``fixed_model`` (additive): append every sample with ``add_sample_fixed`` -- installed hyper-parameters and
    normalisation kept, the next step updates the grid posterior instead of recomputing it (not with ``hypopt``).
    Returns the reference's ``data`` dict: i, obj, con, x_0, x_1 (+ per-iteration info)."""
    _check_append_mode(hypopt, fixed_model)
    data = {"i": [], "obj": [], "con": [], "x_0": [], "x_1": [], "info": []}
    for i in range(n_iteration):
        x_new, info = safeopt_iteration(GP_m, require_lipschitz_ucb)
        plant_output = GP_m.calculate_plant_outputs(x_new, noise)
        data["i"].append(i)
        data["obj"].append(plant_output[0])
        data["con"].append(plant_output[1] if len(plant_output) > 1 else np.nan)
        data["x_0"].append(x_new[0])
        data["x_1"].append(x_new[1] if x_new.shape[0] > 1 else np.nan)
        data["info"].append(info)
        if on_iteration is not None:
            on_iteration(i, GP_m, x_new, plant_output, info)
        _append(GP_m, x_new, plant_output, hypopt, fixed_model)
        if info["std_expander"] < stop_std and info["std_minimizer"] < stop_std:       # :178
            break
    return data


def safeopt_batch_iteration(GP_m, q):
    """One batch acquisition of SafeOpt: q safe points for parallel experiments (BO.Batch).  Pick 1 is safeopt_iteration's
    x_new; the others follow the same rule with the earlier picks as pending observations.  Returns (X (m, d), info)."""
    t0 = time.perf_counter()
    X, std, info = GP_m.Batch(q)
    info = dict(info, std=np.asarray(std), acquisition_seconds=time.perf_counter() - t0)
    if len(X) == 0:
        raise EmptySafeSet("SafeOpt batch: the safe set is empty on the grid (no minimiser and no expander)")
    return np.asarray(X, dtype=np.float64), info


def run_safeopt_batch(GP_m, q, n_iteration=10, noise=0., stop_std=0.01, on_iteration=None, hypopt=None):
    """run_safeopt with q experiments per iteration: each iteration takes a batch of q safe points, evaluates the q plants
    and adds the samples one by one with ``add_sample``; it stops like run_safeopt, on the stds of pick 1 (the step's own
    minimiser and expander).  Returns the dict of run_safeopt with one row per evaluated point plus ``batch`` (the
    iteration of each row) and one ``info`` per iteration."""
    data = {"i": [], "batch": [], "obj": [], "con": [], "x_0": [], "x_1": [], "info": []}
    row = 0
    for it in range(n_iteration):
        X, info = safeopt_batch_iteration(GP_m, q)
        outputs = [GP_m.calculate_plant_outputs(x, noise) for x in X]
        for x, y in zip(X, outputs):
            data["i"].append(row)
            data["batch"].append(it)
            data["obj"].append(y[0])
            data["con"].append(y[1] if len(y) > 1 else np.nan)
            data["x_0"].append(x[0])
            data["x_1"].append(x[1] if x.shape[0] > 1 else np.nan)
            row += 1
        data["info"].append(info)
        if on_iteration is not None:
            on_iteration(it, GP_m, X, outputs, info)
        for x, y in zip(X, outputs):
            if hypopt is None:
                GP_m.add_sample(x, y)
            else:
                GP_m.add_sample(x, y, hypopt=hypopt)
        if info["std_expander"] < stop_std and info["std_minimizer"] < stop_std:
            break
    return data


def run_goose(GP_m, n_iteration=10, noise=0., f_opt=0.145249, tol=0.005, on_iteration=None, hypopt=None,
              fixed_model=False):
    """test/test_GoOSE.py:142-190 without the plotting side effects; stops when the noiseless objective at x_new is
    within ``tol`` of ``f_opt`` (``:182``; pass f_opt=None to run all iterations).  ``hypopt`` and ``fixed_model`` as in
    run_safeopt."""
    _check_append_mode(hypopt, fixed_model)
    data = {"i": [], "obj": [], "con": [], "x_0": [], "x_1": [], "x_target_0": [], "x_target_1": [], "info": []}
    for i in range(n_iteration):
        x_new, info = goose_iteration(GP_m)
        plant_output = GP_m.calculate_plant_outputs(x_new, noise)
        data["i"].append(i)
        data["obj"].append(plant_output[0])
        data["con"].append(plant_output[1] if len(plant_output) > 1 else np.nan)
        data["x_0"].append(x_new[0])
        data["x_1"].append(x_new[1] if x_new.shape[0] > 1 else np.nan)
        data["x_target_0"] = info["x_target"][0]                                       # :172-173 (sic: overwritten)
        data["x_target_1"] = info["x_target"][1] if info["x_target"].shape[0] > 1 else np.nan
        data["info"].append(info)
        if on_iteration is not None:
            on_iteration(i, GP_m, x_new, plant_output, info)
        _append(GP_m, x_new, plant_output, hypopt, fixed_model)
        if f_opt is not None and abs(GP_m.plant_system[0](x_new) - f_opt) <= tol:
            break
    return data


def goose_batch_iteration(GP_m, q):
    """One batch acquisition of GoOSE: q distinct safe points for parallel experiments (BO.Batch).  Pick 1 is
    goose_iteration's x_new; the others follow the same rule over the safe points and targets not yet used, with the
    earlier picks as pending observations.  Returns (X (m, d), info)."""
    t0 = time.perf_counter()
    X, lcb, info = GP_m.Batch(q)
    info = dict(info, lcb=np.asarray(lcb), acquisition_seconds=time.perf_counter() - t0)
    if len(X) == 0:
        raise EmptySafeSet("GoOSE batch: the safe set is empty on the grid (no safe minimum and no reachable target)")
    return np.asarray(X, dtype=np.float64), info


def run_goose_batch(GP_m, q, n_iteration=10, noise=0., f_opt=0.145249, tol=0.005, on_iteration=None, hypopt=None):
    """run_goose with q experiments per iteration: each iteration takes a batch of q safe points, evaluates the q plants
    and adds the samples one by one with ``add_sample``; it stops like run_goose, when the noiseless objective at pick 1
    (the step's own x_new) is within ``tol`` of ``f_opt`` (f_opt=None runs all iterations).  Returns the dict of run_goose
    with one row per evaluated point plus ``batch`` (the iteration of each row) and one ``info`` per iteration."""
    data = {"i": [], "batch": [], "obj": [], "con": [], "x_0": [], "x_1": [], "x_target_0": [], "x_target_1": [], "info": []}
    row = 0
    for it in range(n_iteration):
        X, info = goose_batch_iteration(GP_m, q)
        outputs = [GP_m.calculate_plant_outputs(x, noise) for x in X]
        for x, y, xt in zip(X, outputs, info["x_target"]):
            data["i"].append(row)
            data["batch"].append(it)
            data["obj"].append(y[0])
            data["con"].append(y[1] if len(y) > 1 else np.nan)
            data["x_0"].append(x[0])
            data["x_1"].append(x[1] if x.shape[0] > 1 else np.nan)
            data["x_target_0"].append(xt[0])
            data["x_target_1"].append(xt[1] if xt.shape[0] > 1 else np.nan)
            row += 1
        data["info"].append(info)
        if on_iteration is not None:
            on_iteration(it, GP_m, X, outputs, info)
        for x, y in zip(X, outputs):
            if hypopt is None:
                GP_m.add_sample(x, y)
            else:
                GP_m.add_sample(x, y, hypopt=hypopt)
        if f_opt is not None and abs(GP_m.plant_system[0](X[0]) - f_opt) <= tol:
            break
    return data


def run_multiple(make_bo, x_init, r, n_sample, n_start, n_iteration, noise, algorithm="safeopt", path=None,
                 stop_std=0.01, seeds=None):
    """test/test_SafeOpt.py:188-253 / :255-322 and the GoOSE counterparts: ``n_start`` independent runs, each
    starting from ``n_sample`` points drawn in the ball (x_init, r), recorded in the reference's layout.
    ``make_bo()`` returns a fresh BO object; ``seeds[i]`` (optional) seeds run i (sampling and hyper-fit).
    Writes ``path`` (npz) if given and returns the dict."""
    data = {}
    for i in range(n_start):
        GP_m = make_bo()
        if seeds is not None:
            GP_m.key = np.random.default_rng(int(seeds[i]))
            GP_m.hyper_seed = int(seeds[i])
        X, Y = GP_m.Data_sampling(n_sample, np.asarray(x_init, dtype=np.float64), r, noise)
        GP_m.GP_initialization(X, Y, 'RBF', multi_hyper=5, var_out=True)
        run = {"sampled_x": np.asarray(X), "sampled_output": np.asarray(Y), "observed_x": [], "observed_output": []}
        for _ in range(n_iteration):
            if algorithm == "safeopt":
                x_new, info = safeopt_iteration(GP_m, require_lipschitz_ucb=True)
            else:
                x_new, info = goose_iteration(GP_m)
            plant_output = GP_m.calculate_plant_outputs(x_new, noise)
            GP_m.add_sample(x_new, plant_output)
            run["observed_x"].append(np.asarray(x_new))
            run["observed_output"].append(np.asarray(plant_output))
            if algorithm == "safeopt" and info["std_expander"] < stop_std and info["std_minimizer"] < stop_std:
                break
        run["observed_x"] = np.array(run["observed_x"])
        run["observed_output"] = np.array(run["observed_output"])
        data[f"{i}"] = run
    if path is not None:
        save_runs(path, data)
    return data


def save_runs(path, data):
    """``jnp.savez('data/...npz', **data)`` of the reference (test_SafeOpt.py:253) with NumPy arrays."""
    np.savez(path, **{k: np.array(v, dtype=object) for k, v in data.items()})


def load_runs(path):
    """Read a result file written by save_runs (or by the reference, if its arrays unpickle): {run: dict}."""
    with np.load(path, allow_pickle=True) as z:
        return {k: z[k].item() for k in z.files}
