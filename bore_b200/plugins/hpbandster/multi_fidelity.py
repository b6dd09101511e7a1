"""Multi-fidelity HpBandSter plugin: one recurrent classifier over the rungs of Hyperband
(same surface as bore/plugins/hpbandster/multi_fidelity.py:19-329: ``BOREHyperband``,
``SequenceClassifierConfigGenerator``).

Every configuration is a sequence over the budgets it has been evaluated at; the stacked-LSTM
classifier (``bore_b200.recurrent``, csrc/lstm.cu) is trained many-to-many on those padded sequences,
and a proposal maximises the one-to-one view of the same weights at the highest rung that already
holds ``num_random_init`` evaluations.  The order in which ``config_space``'s RNG and
``self.random_state`` are consumed follows the reference call by call.

One deliberate difference: ``mask_value`` is read from ``classifier_kws`` with the reference's
``BOREHyperband`` default (-1.0) when the key is missing -- the reference's generator falls back to
1e-9 there (multi_fidelity.py:112), a value its own front end never passes.
"""
import logging

import numpy as np

from ._compat import HyperBand, base_config_generator
from .base import TRANSFORMS
from .types import DenseConfigurationSpace, array_from_dict, dict_from_array
from ...base import maybe_distort
from ...data import MultiFidelityRecord, UniqueFilter
from ...layers import BinaryCrossentropy, l2, optimizer_spec
from ...math import steps_per_epoch
from ...models import StackedRecurrentFactory


class BOREHyperband(HyperBand):
    """Hyperband driven by ``SequenceClassifierConfigGenerator`` (multi_fidelity.py:19-85)."""

    def __init__(self, config_space, eta=3, min_budget=0.01, max_budget=1,
                 gamma=None, num_random_init=10, random_rate=0.1, retrain=False,
                 num_starts=5, num_samples=1024, batch_size=64,
                 num_steps_per_iter=1000, num_epochs=None, optimizer="adam",
                 mask_value=-1.,
                 num_layers=2, num_units=32, activation="elu", l2_factor=None,
                 transform="sigmoid", method="L-BFGS-B", max_iter=1000,
                 ftol=1e-9, distortion=None, seed=None, device=None, **kwargs):
        gamma = 1 / eta if gamma is None else gamma
        classifier = dict(num_layers=num_layers, num_units=num_units, l2_factor=l2_factor,
                          activation=activation, optimizer=optimizer, mask_value=mask_value)
        training = dict(batch_size=batch_size, num_steps_per_iter=num_steps_per_iter, num_epochs=num_epochs)
        acquisition = dict(transform=transform, method=method, max_iter=max_iter, ftol=ftol,
                           distortion=distortion, num_starts=num_starts, num_samples=num_samples)
        generator = SequenceClassifierConfigGenerator(
            config_space=config_space, gamma=gamma, num_random_init=num_random_init,
            random_rate=random_rate, retrain=retrain, classifier_kws=classifier, fit_kws=training,
            optimizer_kws=acquisition, seed=seed, device=device)
        # the GRANDPARENT initializer, as in the reference: Hyperband's own sampler is never built
        super(HyperBand, self).__init__(config_generator=generator, **kwargs)

        self.eta, self.min_budget, self.max_budget = eta, min_budget, max_budget
        self.max_SH_iter = -int(np.log(min_budget / max_budget) / np.log(eta)) + 1
        self.budgets = max_budget * np.power(
            eta, -np.linspace(self.max_SH_iter - 1, 0, self.max_SH_iter))
        self.config.update(dict(eta=eta, min_budget=min_budget, max_budget=max_budget,
                                budgets=self.budgets, max_SH_iter=self.max_SH_iter, gamma=gamma,
                                num_random_init=num_random_init, seed=seed))


class SequenceClassifierConfigGenerator(base_config_generator):

    def __init__(self, config_space, gamma, num_random_init, random_rate,
                 retrain, classifier_kws, fit_kws, optimizer_kws, seed, device=None, **kwargs):
        super(SequenceClassifierConfigGenerator, self).__init__(**kwargs)

        assert 0. < gamma < 1., "`gamma` must be in (0, 1)"
        assert num_random_init > 0, "number of initial random designs must be non-zero!"
        assert random_rate is None or 0. <= random_rate < 1., "`random_rate` must be in [0, 1)"
        if retrain:
            raise NotImplementedError  # as the reference (multi_fidelity.py:136-137)
        self.gamma, self.num_random_init, self.random_rate = gamma, num_random_init, random_rate
        self.retrain = retrain

        # dense one-hot view of the space: the classifier sees the unit cube
        self.config_space = DenseConfigurationSpace(config_space, seed=seed)
        self.input_dim = self.config_space.get_dimensions(sparse=False)
        self.bounds = self.config_space.get_bounds()

        # classifier
        self.optimizer = classifier_kws.get("optimizer", "adam")
        optimizer_spec(self.optimizer, "BOREHyperband")  # refused here, not at the first fit
        self.mask_value = classifier_kws.get("mask_value", -1.)
        factor = classifier_kws.get("l2_factor")
        penalty = None if factor is None else l2(factor)
        self.model_factory = StackedRecurrentFactory(
            input_dim=self.input_dim, output_dim=1,
            num_layers=classifier_kws.get("num_layers", 2),
            num_units=classifier_kws.get("num_units", 32),
            layer_kws=dict(activation=classifier_kws.get("activation", "elu"),
                           kernel_regularizer=penalty, bias_regularizer=penalty),
            seed=None if seed is None else seed + 1, device=device)
        self.logit = self._build_compile_network()
        self.funcs = {}  # rung -> one-to-one network, built on first use

        # training
        self.batch_size = fit_kws.get("batch_size", 64)
        self.num_steps_per_iter = fit_kws.get("num_steps_per_iter", 100)
        self.num_epochs = fit_kws.get("num_epochs")

        # acquisition maximisation
        name = optimizer_kws.get("transform", "sigmoid")
        assert name in TRANSFORMS, f"`transform` must be one of {tuple(TRANSFORMS.keys())}"
        self.transform = TRANSFORMS.get(name)
        assert optimizer_kws.get("num_starts") > 0
        self.num_starts = optimizer_kws.get("num_starts", 5)
        self.num_samples = optimizer_kws.get("num_samples", 1024)
        self.method = optimizer_kws.get("method", "L-BFGS-B")
        self.ftol = optimizer_kws.get("ftol", 1e-9)
        self.max_iter = optimizer_kws.get("max_iter", 1000)
        self.distortion = optimizer_kws.get("distortion")

        self.record = MultiFidelityRecord(gamma=gamma)
        self.seed = seed
        self.random_state = np.random.RandomState(seed)

    # ------------------------------------------------------------------ classifier
    def _build_compile_network(self):
        self.logger.debug("Building and compiling network...")
        network = self.model_factory.build_many_to_many(mask_value=self.mask_value)
        network.compile(optimizer=self.optimizer, metrics=["accuracy"],
                        loss=BinaryCrossentropy(from_logits=True))
        network.summary(print_fn=self.logger.debug)
        return network

    def _update_classifier(self):
        inputs, targets = self.record.sequences(binary=True, pad_value=self.mask_value)
        self.logger.debug(f"Input sequence shape: {inputs.shape}")
        self.logger.debug(f"Target sequence shape: {targets.shape}")

        num_steps = steps_per_epoch(self.record.num_features(), self.batch_size)
        if self.num_epochs is None:
            num_epochs = self.num_steps_per_iter // num_steps
            self.logger.debug("Argument `num_epochs` has not been specified. "
                              f"Setting num_epochs={num_epochs}")
        else:
            num_epochs = self.num_epochs
            self.logger.debug(f"Argument `num_epochs` is specified (num_epochs={num_epochs}). "
                              f"Ignoring num_steps_per_iter={self.num_steps_per_iter}")

        self.logit.fit(inputs, targets, epochs=num_epochs, batch_size=self.batch_size,
                       callbacks=[], verbose=False)
        loss, accuracy = self.logit.evaluate(inputs, targets, verbose=False)
        self.logger.info(f"[Model fit: loss={loss:.3f}, accuracy={accuracy:.3f}] "
                         f"batch size: {self.batch_size}, "
                         f"num steps per iter: {self.num_steps_per_iter}, "
                         f"num epochs: {num_epochs}")

    def _is_unique(self, res):
        is_duplicate = self.record.is_duplicate(res.x)
        if is_duplicate:
            self.logger.warning("Duplicate detected! Skipping...")
        return not is_duplicate

    @property
    def _print_fn(self):
        """``self.logger.debug`` while DEBUG lines would be emitted (what the reference passes,
        multi_fidelity.py:276), else None so that only the winner leaves the GPU."""
        enabled = getattr(self.logger, "isEnabledFor", None)
        if enabled is not None and not enabled(logging.DEBUG):
            return None
        return self.logger.debug

    # ------------------------------------------------------------------ HpBandSter interface
    def get_config(self, budget):
        fallback = (self.config_space.sample_configuration().get_dictionary(), {})

        # epsilon-greedy exploration
        if self.random_rate is not None and self.random_state.binomial(p=self.random_rate, n=1):
            self.logger.info(f"[Glob. maximum: skipped (prob={self.random_rate:.2f})] "
                             "Suggesting random candidate ...")
            return fallback

        # the highest rung that already has enough evaluations decides which output step is maximised
        t = self.record.highest_rung(min_size=self.num_random_init)
        if t is None:
            self.logger.debug(f"There are no rungs with at least {self.num_random_init} observations. "
                              "Suggesting random candidate...")
            return fallback
        self.logger.debug(f"Rung {t} is the highest with at least {self.num_random_init} observations.")

        self._update_classifier()

        # rungs are zero-based: rung t reads the output of step t + 1
        if t not in self.funcs:
            self.funcs[t] = self.model_factory.build_one_to_one(t + 1, transform=self.transform)
        func = self.funcs[t]

        self.logger.debug(f"Beginning multi-start maximization with {self.num_starts} starts...")
        opt = func.argmax(self.bounds, num_starts=self.num_starts, num_samples=self.num_samples,
                          method=self.method, options=dict(maxiter=self.max_iter, ftol=self.ftol),
                          print_fn=self._print_fn, filter_fn=UniqueFilter(self.record, logger=self.logger),
                          random_state=self.random_state)
        if opt is None:
            self.logger.warning("[Glob. maximum: not found!] Either optimization "
                                f"failed in all {self.num_starts} starts, or "
                                "all maxima found have been evaluated previously!"
                                " Suggesting random candidate...")
            return fallback

        self.logger.info(f"[Glob. maximum: value={-opt.fun:.3f} x={opt.x}]")
        suggestion = maybe_distort(opt.x, self.distortion, self.bounds, self.random_state,
                                   print_fn=self.logger.info)
        return (dict_from_array(self.config_space, suggestion), {})

    def new_result(self, job, update_model=True):
        super(SequenceClassifierConfigGenerator, self).new_result(job)
        budget = job.kwargs["budget"]
        x = array_from_dict(self.config_space, job.kwargs["config"])
        self.record.append(x=x, y=job.result["loss"], b=budget)
        self.logger.debug(f"[Data] rungs: {self.record.num_rungs()}, budgets: {self.record.budgets()}, "
                          f"rung sizes: {self.record.rung_sizes()}")
        self.logger.debug(f"[Data] thresholds: {self.record.thresholds()}")
