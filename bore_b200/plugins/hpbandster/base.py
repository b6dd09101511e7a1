"""HpBandSter config generator driving the B200 hot path (same surface as
bore/plugins/hpbandster/base.py:21-288: ``BORE``, ``ClassifierConfigGenerator``, ``TRANSFORMS``).

``get_config(budget)`` is the named caller of the path: epsilon-greedy / warm-up gates, then
``fit`` (fused CUDA training kernel) on the quantile-labelled record and ``argmax`` (on-device
multi-start L-BFGS-B) over the dense unit cube, duplicate filter, optional distortion, decode.
The order in which ``self.random_state`` and the config space's RNG are consumed follows the
reference call by call (sample a random config first, then the binomial, then -- inside
``argmax`` -- the uniform start points, then the optional truncated normal), so a replay with
the same seed proposes the same sequence of gates.

Build extension (BASELINE.json configs[4]): ``per_budget=True`` keeps one record and one
classifier per Hyperband budget instead of pooling all observations (the reference's MLP
generator ignores the budget, base.py:280); a proposal for budget b uses the classifier of the
largest budget <= b that already has ``num_random_init`` observations, BOHB-style.

HpBandSter and ConfigSpace are used when installed, else the stand-ins in ``_compat``.
"""
import logging

import numpy as np

from ._compat import HyperBand, base_config_generator
from .types import DenseConfigurationSpace, array_from_dict, dict_from_array
from ... import ops
from ...base import maybe_distort
from ...data import Record, UniqueFilter
from ...layers import BinaryCrossentropy, activation_name, l2, optimizer_spec
from ...math import steps_per_epoch
from ...models import MaximizableDenseSequential

TRANSFORMS = dict(identity=ops.identity, sigmoid=ops.sigmoid, exp=ops.exp)


class BORE(HyperBand):
    """Hyperband whose config sampler is the BORE classifier (plugins/hpbandster/base.py:21-81)."""

    def __init__(self, config_space, eta=3, min_budget=0.01, max_budget=1,
                 gamma=None, num_random_init=10, random_rate=0.1, retrain=False,
                 num_starts=5, num_samples=1024, batch_size=64,
                 num_steps_per_iter=1000, num_epochs_per_iter=None,
                 optimizer="adam",
                 num_layers=2, num_units=32, activation="elu", l2_factor=None,
                 transform="sigmoid", method="L-BFGS-B", max_iter=1000,
                 ftol=1e-9, distortion=None, seed=None, per_budget=False, device=None, **kwargs):
        gamma = 1 / eta if gamma is None else gamma
        generator = ClassifierConfigGenerator(
            config_space=config_space, gamma=gamma, num_random_init=num_random_init,
            random_rate=random_rate, retrain=retrain,
            classifier_kws=dict(num_layers=num_layers, num_units=num_units, l2_factor=l2_factor,
                                activation=activation, optimizer=optimizer),
            fit_kws=dict(batch_size=batch_size, num_steps_per_iter=num_steps_per_iter,
                         num_epochs_per_iter=num_epochs_per_iter),
            optimizer_kws=dict(transform=transform, method=method, max_iter=max_iter, ftol=ftol,
                               distortion=distortion, num_starts=num_starts,
                               num_samples=num_samples),
            seed=seed, per_budget=per_budget, device=device)
        # as in the reference: the GRANDPARENT initializer, so that Hyperband's own (random)
        # config generator is never built
        super(HyperBand, self).__init__(config_generator=generator, **kwargs)

        # Hyperband's bracket arithmetic
        self.eta, self.min_budget, self.max_budget = eta, min_budget, max_budget
        self.max_SH_iter = -int(np.log(min_budget / max_budget) / np.log(eta)) + 1
        self.budgets = max_budget * np.power(
            eta, -np.linspace(self.max_SH_iter - 1, 0, self.max_SH_iter))
        self.config.update(dict(eta=eta, min_budget=min_budget, max_budget=max_budget,
                                budgets=self.budgets, max_SH_iter=self.max_SH_iter, gamma=gamma,
                                num_random_init=num_random_init, seed=seed))


class ClassifierConfigGenerator(base_config_generator):

    def __init__(self, config_space, gamma, num_random_init, random_rate,
                 retrain, classifier_kws, fit_kws, optimizer_kws, seed, per_budget=False,
                 device=None, **kwargs):
        super(ClassifierConfigGenerator, self).__init__(**kwargs)

        assert 0. < gamma < 1., "`gamma` must be in (0, 1)"
        assert num_random_init > 0, "number of initial random designs must be non-zero!"
        assert random_rate is None or 0. <= random_rate < 1., "`random_rate` must be in [0, 1)"
        self.gamma, self.num_random_init, self.random_rate = gamma, num_random_init, random_rate

        # one-hot dense view of the space; the classifier lives on its unit cube
        self.config_space = DenseConfigurationSpace(config_space, seed=seed)
        self.input_dim = self.config_space.get_dimensions(sparse=False)
        self.bounds = self.config_space.get_bounds()

        # classifier
        self.num_layers = classifier_kws.get("num_layers", 2)
        self.num_units = classifier_kws.get("num_units", 32)
        self.activation = activation_name(classifier_kws.get("activation", "elu"), "BORE")
        self.optimizer = classifier_kws.get("optimizer", "adam")
        optimizer_spec(self.optimizer, "BORE")  # refused here, not at the first fit
        l2_factor = classifier_kws.get("l2_factor")
        self.kernel_regularizer = None if l2_factor is None else l2(l2_factor)
        self.bias_regularizer = None if l2_factor is None else l2(l2_factor)
        self.retrain = retrain
        self.logit = None
        self.device = device

        # training
        self.batch_size = fit_kws.get("batch_size", 64)
        self.num_steps_per_iter = fit_kws.get("num_steps_per_iter", 100)
        self.num_epochs_per_iter = fit_kws.get("num_epochs_per_iter")

        # acquisition maximisation
        transform_name = optimizer_kws.get("transform", "sigmoid")
        assert transform_name in TRANSFORMS, \
            f"`transform` must be one of {tuple(TRANSFORMS.keys())}"
        self.transform = TRANSFORMS.get(transform_name)
        self.num_starts = optimizer_kws.get("num_starts")
        self.num_samples = optimizer_kws.get("num_samples", 1024)
        self.method = optimizer_kws.get("method", "L-BFGS-B")
        self.ftol = optimizer_kws.get("ftol", 1e-9)
        self.max_iter = optimizer_kws.get("max_iter", 1000)
        self.distortion = optimizer_kws.get("distortion")

        self.record = Record()
        self.seed = seed
        self.random_state = np.random.RandomState(seed)

        # build extension: one (record, classifier) pair per budget
        self.per_budget = bool(per_budget)
        self._budget_records = {}
        self._budget_logits = {}

    # ------------------------------------------------------------------ classifier lifecycle
    def _build_compile_network(self):
        self.logger.debug("Building and compiling network...")
        network = MaximizableDenseSequential(
            transform=self.transform, input_dim=self.input_dim, output_dim=1,
            num_layers=self.num_layers, num_units=self.num_units,
            layer_kws=dict(activation=self.activation,
                           kernel_regularizer=self.kernel_regularizer,
                           bias_regularizer=self.bias_regularizer),
            seed=None if self.seed is None else self.seed + 1, device=self.device)
        network.compile(optimizer=self.optimizer, metrics=["accuracy"],
                        loss=BinaryCrossentropy(from_logits=True))
        network.summary(print_fn=self.logger.debug)
        return network

    def _maybe_create_classifier(self):
        if self.logit is None:
            self.logit = self._build_compile_network()

    def _maybe_delete_classifier(self):
        if self.retrain:  # train from scratch at the next proposal
            self.logger.debug("Deleting model...")
            self.logit = None

    def _update_classifier(self):
        X, z = self.record.load_classification_data(self.gamma)
        dataset_size = self.record.size()
        num_steps = steps_per_epoch(dataset_size, self.batch_size)

        num_epochs_per_iter = self.num_epochs_per_iter
        if num_epochs_per_iter is None:
            num_epochs_per_iter = self.num_steps_per_iter // num_steps
            self.logger.debug("Argument `num_epochs_per_iter` has not been specified. "
                              f"Setting num_epochs_per_iter={num_epochs_per_iter}")
        else:
            self.logger.debug("Argument `num_epochs_per_iter` is specified "
                              f"(num_epochs_per_iter={num_epochs_per_iter}). "
                              f"Ignoring num_steps_per_iter={self.num_steps_per_iter}")

        self.logit.fit(X, z, epochs=num_epochs_per_iter, batch_size=self.batch_size,
                       callbacks=[], verbose=False)
        loss, accuracy = self.logit.evaluate(X, z, verbose=False)
        self.logger.info(f"[Model fit: loss={loss:.3f}, accuracy={accuracy:.3f}] "
                         f"dataset size: {dataset_size}, batch size: {self.batch_size}, "
                         f"steps per epoch: {num_steps}, "
                         f"num steps per iter: {self.num_steps_per_iter}, "
                         f"num epochs: {num_epochs_per_iter}")

    @property
    def _print_fn(self):
        """``print_fn=self.logger.debug`` as the reference passes it
        (bore/plugins/hpbandster/base.py:263) -- but only while the logger would emit the
        per-start lines; otherwise None, so that only the winner leaves the GPU."""
        enabled = getattr(self.logger, "isEnabledFor", None)
        if enabled is not None and not enabled(logging.DEBUG):
            return None
        return self.logger.debug

    def _unique_filter(self):
        """The reference passes ``filter_fn=self._is_unique`` (one Python callback per result);
        ``UniqueFilter`` is the same predicate in a form ``argmax`` can evaluate for all results
        in one launch when nothing has to be printed per start."""
        return UniqueFilter(self.record, logger=self.logger)

    def _is_unique(self, res):
        is_duplicate = self.record.is_duplicate(res.x)
        if is_duplicate:
            self.logger.warning("Duplicate detected! Skipping...")
        return not is_duplicate

    # ------------------------------------------------------------------ per-budget extension
    def _select_budget(self, budget):
        """Largest observed budget <= ``budget`` (else largest overall) whose record already
        holds ``num_random_init`` observations; None if there is none."""
        ready = sorted(b for b, r in self._budget_records.items()
                       if r.size() >= self.num_random_init)
        if not ready:
            return None
        below = [b for b in ready if b <= budget]
        return below[-1] if below else ready[-1]

    def _bind_budget(self, b):
        self.record = self._budget_records[b]
        self.logit = self._budget_logits.get(b)

    # ------------------------------------------------------------------ HpBandSter interface
    def get_config(self, budget):
        config_random = self.config_space.sample_configuration()
        config_random_dict = config_random.get_dictionary()

        # epsilon-greedy exploration
        if self.random_rate is not None and self.random_state.binomial(p=self.random_rate, n=1):
            self.logger.info(f"[Glob. maximum: skipped (prob={self.random_rate:.2f})] "
                             "Suggesting random candidate ...")
            return (config_random_dict, {})

        if self.per_budget:
            b = self._select_budget(budget)
            if b is None:
                self.logger.debug("No budget has completed its initial runs yet. "
                                  "Suggesting random candidate...")
                return (config_random_dict, {})
            self._bind_budget(b)

        # insufficient training data
        dataset_size = self.record.size()
        if dataset_size < self.num_random_init:
            self.logger.debug(f"Completed {dataset_size}/{self.num_random_init}"
                              " initial runs. Suggesting random candidate...")
            return (config_random_dict, {})

        self._maybe_create_classifier()
        self._update_classifier()

        self.logger.debug(f"Beginning multi-start maximization with {self.num_starts} starts...")
        opt = self.logit.argmax(self.bounds, num_starts=self.num_starts,
                                num_samples=self.num_samples, method=self.method,
                                options=dict(maxiter=self.max_iter, ftol=self.ftol),
                                print_fn=self._print_fn, filter_fn=self._unique_filter(),
                                random_state=self.random_state)
        if self.per_budget:
            self._budget_logits[b] = None if self.retrain else self.logit
        if opt is None:
            self.logger.warning("[Glob. maximum: not found!] Either optimization "
                                f"failed in all {self.num_starts} starts, or "
                                "all maxima found have been evaluated previously!"
                                " Suggesting random candidate...")
            return (config_random_dict, {})

        loc = opt.x
        self.logger.info(f"[Glob. maximum: value={-opt.fun:.3f} x={loc}]")
        config_opt_arr = maybe_distort(loc, self.distortion, self.bounds, self.random_state,
                                       print_fn=self.logger.info)
        config_opt_dict = dict_from_array(self.config_space, config_opt_arr)
        self._maybe_delete_classifier()
        return (config_opt_dict, {})

    def new_result(self, job, update_model=True):
        super(ClassifierConfigGenerator, self).new_result(job)
        budget = job.kwargs["budget"]
        config_arr = array_from_dict(self.config_space, job.kwargs["config"])
        loss = job.result["loss"]
        if self.per_budget:
            self._budget_records.setdefault(budget, Record()).append(x=config_arr, y=loss, b=budget)
        else:
            # the pooled record ignores the budget, as the reference does
            self.record.append(x=config_arr, y=loss, b=budget)
