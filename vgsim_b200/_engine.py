"""Host side of the engine: the object that sits behind ``Simulator.simulation``.

This is the drop-in replacement for the reference's ``cdef class BirthDeathModel``
(reference ``src/_BirthDeath.pyx:30-2649``) at the boundary SURVEY.md §8(b) describes:
same constructor arguments, same ``set_*`` methods / read-only properties (live numpy views),
same exception types and messages, same ``SimulatePopulation`` / ``SimulatePopulation_tau`` /
``GetGenealogy`` entry points.  The parameter store and validation are plain Python + numpy; the
hot path (forward simulation, genealogy) runs in hand-written sm_100a CUDA kernels reached through
the C ABI of ``libvgsim_b200.so`` (``include/vgsim_b200.h``).  There is no CPU fallback: without the
library or without a GPU the hot-path calls raise.

Extension over the reference: ``replicates=R`` runs R independent replicates (replicate ``r`` uses
seed ``seed + r``) in one batched launch; with the default ``R == 1`` the object behaves like the
reference engine.  Outputs take a ``replicate=`` index.
"""
import sys

import numpy as np

from . import _capi
from . import _params as P

_GENOME_TEXT = ('Incorrect value of number of sites or genome length. Genome length should be more or equal number of sites.')


_RECOMB_TEXT = ('recombination / coinfection (recombination_probability > 0) is out of scope of the device path: the forward '
                'kernels do not generate recombinant births')


def _warn_recombination(probability):
    """The reference's Birth() takes its recombination branch whenever rn < recombination_probability
    (src/_BirthDeath.pyx:575-596).  That experimental branch (SURVEY 2 #6: logs one haplotype, infects another, ignored by
    the genealogy) is not part of the device path.  The value is stored (the reference's interface tests read it back),
    setting it warns, and simulate() refuses to run with it instead of silently producing a non-recombinant run."""
    if probability > 0:
        import warnings
        warnings.warn(_RECOMB_TEXT + '; simulate() will raise NotImplementedError', stacklevel=3)


BIRTH, DEATH, SAMPLING, MUTATION, SUSCCHANGE, MIGRATION, MULTITYPE = range(7)  # src/events.pxi:2-8


class BirthDeathModel:
    # ------------------------------------------------------------------ construction (src/_BirthDeath.pyx:70-229)
    def __init__(self, number_of_sites, populations_number, number_of_susceptible_groups, seed,
                 sampling_probability, memory_optimization, genome_length, recombination_probability,
                 replicates=1, device=None):
        P.count(seed, 'seed', positive=False)
        self.user_seed = seed
        self.first_simulation = False
        for flag, what in ((sampling_probability, 'sampling probability'), (memory_optimization, 'memory optimization')):
            if flag != True and flag != False:  # noqa: E712  (0 / 1 are accepted like the reference does)
                raise ValueError('Incorrect value of %s. Value of %s should be True or False.' % (what, what))
        self._sampling_probability = sampling_probability
        self._memory_optimization = memory_optimization

        self.sites = P.count(number_of_sites, 'number of sites', positive=False)
        self.hapNum = int(4 ** self.sites)
        self.susNum = P.count(number_of_susceptible_groups, 'number of susceptible groups')
        self.popNum = P.count(populations_number, 'populations number')
        self._haps = P.Axis(self.hapNum, 'haplotype', sites=self.sites)
        self._demes = P.Axis(self.popNum, 'population')
        self._groups = P.Axis(self.susNum, 'susceptibility type')
        self._sites_axis = P.Axis(self.sites, 'mutation site')

        self.recombination = P.quantity(recombination_probability, 'recombination probability', upper=1)
        _warn_recombination(recombination_probability)
        self._genome_length = P.count(genome_length, 'genome length')
        self.sitesPosition = np.zeros(self.sites, dtype=np.int64)
        if self.sites > self._genome_length:
            raise ValueError(_GENOME_TEXT)
        if self.sites > 1:
            self._place_sites()

        # memory optimisation (lazy haplotype slots, SURVEY §2 #5) is a direct-method-only CPU memory
        # trick; the device path keeps the dense K x H state.  The knobs are kept for API compatibility.
        if self._memory_optimization:
            if self.sites > 2:
                self.maxHapNum = int(4 ** (self.sites - 2))
                self.addMemoryNum = int(4 ** (self.sites - 2))
            else:
                self.maxHapNum = 4
                self.addMemoryNum = 4
        else:
            self.maxHapNum = self.hapNum
            self.addMemoryNum = 0

        H, K, S, U = self.hapNum, self.popNum, self.susNum, self.sites
        self.suscType = np.zeros(H, dtype=np.int64)
        self.bRate = np.full(H, 2.0)
        self.dRate = np.full(H, 1.0)
        self.sRate = np.full(H, 0.01)
        self.mRate = np.full((H, U), 0.01)
        self._susceptibility = np.zeros((H, S), dtype=float)
        self._susceptibility[:, 0] = 1.0
        self.hapMutType = np.ones((H, U, 3), dtype=float)

        self.sizes = np.full(K, 1000000, dtype=np.int64)
        self._susceptible = np.zeros((K, S), dtype=np.int64)
        self._susceptible[:, 0] = 1000000
        self._infectious = np.zeros((K, H), dtype=np.int64)
        self.contactDensity = np.ones(K, dtype=float)
        self.contactDensityBeforeLockdown = np.ones(K, dtype=float)
        self.contactDensityAfterLockdown = np.zeros(K, dtype=float)
        self.startLD = np.ones(K, dtype=float)
        self.endLD = np.ones(K, dtype=float)
        self.samplingMultiplier = np.ones(K, dtype=float)
        self.suscepTransition = np.zeros((S, S), dtype=float)
        self.migrationRates = np.zeros((K, K), dtype=float)

        self.replicates = P.count(replicates, 'replicates')
        self._cd_touched = np.ones(K, dtype=bool)   # demes whose live contact density the next upload overwrites
        self._device = device
        self._handle = None
        self._dirty = True  # parameters changed since last upload
        self._genealogy_done = False
        self.last_elapsed = None

    # ------------------------------------------------------------------ axes and haplotype words
    # (validation and index selection live in _params.py; the behaviour is the reference's setter layer,
    #  src/_BirthDeath.pyx:1187-1702, as pinned by its 278 interface tests)
    def calculate_string_from_haplotype(self, haplotype):
        return self._haps.decode(haplotype)

    calculate_string = calculate_string_from_haplotype  # the name the reference's printing code expects (Q12)

    def calculate_haplotype_from_string(self, string):
        return self._haps.encode(string)

    def create_list_for_cycles(self, index, edge):
        axis = self._haps if edge == self.hapNum else P.Axis(edge, 'index')
        return [int(i) for i in axis.indices(index)]

    # ------------------------------------------------------------------ read-only scalars (:1269-1295)
    seed = property(lambda self: self.user_seed)
    sampling_probability = property(lambda self: self._sampling_probability)
    memory_optimization = property(lambda self: self._memory_optimization)
    number_of_sites = property(lambda self: self.sites)
    haplotypes_number = property(lambda self: self.hapNum)
    haplotype_number = haplotypes_number
    populations_number = property(lambda self: self.popNum)
    number_of_susceptible_groups = property(lambda self: self.susNum)

    # ------------------------------------------------------------------ parameter views (live numpy arrays, like the reference's properties)
    initial_haplotype = property(lambda self: self.maxHapNum)
    step_haplotype = property(lambda self: self.addMemoryNum)
    genome_length = property(lambda self: self._genome_length)
    coinfection_parameters = property(lambda self: self.recombination)
    transmission_rate = property(lambda self: self.bRate)
    recovery_rate = property(lambda self: self.dRate)
    sampling_rate = property(lambda self: self.sRate)
    mutation_rate = property(lambda self: self.mRate)
    mutation_probabilities = property(lambda self: self.hapMutType)
    mutation_position = property(lambda self: self.sitesPosition)
    susceptibility_type = property(lambda self: self.suscType)
    susceptibility = property(lambda self: self._susceptibility)
    immunity_transition = property(lambda self: self.suscepTransition)
    population_size = property(lambda self: self.sizes)
    susceptible = property(lambda self: self._susceptible)
    infectious = property(lambda self: self._infectious)
    contact_density = property(lambda self: self.contactDensity)
    npi = property(lambda self: [self.contactDensityAfterLockdown, self.startLD, self.endLD])
    sampling_multiplier = property(lambda self: self.samplingMultiplier)
    migration_probability = property(lambda self: self.migrationRates)

    def _changed(self):
        self._dirty = True

    def _sites_axis_named(self, what):
        return P.Axis(self.sites, what)

    # ------------------------------------------------------------------ setters
    def _need_memory_optimization(self):
        if not self._memory_optimization:
            raise ValueError("Incorrect value of memory optimization. Value should be equal 'True' for work this function.")

    def set_initial_haplotype(self, amount):
        self._need_memory_optimization()
        P.count(amount, 'amount of initial haplotype')
        self.maxHapNum = min(amount, self.hapNum)

    def set_step_haplotype(self, amount):
        self._need_memory_optimization()
        self.addMemoryNum = P.count(amount, 'amount of step haplotype')

    def _place_sites(self):
        for site in range(self.sites):
            self.sitesPosition[site] = int(site * self._genome_length / (self.sites - 1))

    def set_genome_length(self, genome_length):
        P.count(genome_length, 'genome length')
        if self.sites > genome_length:
            raise ValueError(_GENOME_TEXT)
        self._genome_length = genome_length
        self._place_sites()

    def set_coinfection_parameters(self, recombination):
        self.recombination = P.quantity(recombination, 'recombination probability', upper=1)
        _warn_recombination(recombination)

    def set_transmission_rate(self, rate, haplotype):
        P.quantity(rate, 'transmission rate')
        self.bRate[self._haps.select(haplotype)] = rate
        self._changed()

    def set_recovery_rate(self, rate, haplotype):
        P.quantity(rate, 'recovery rate')
        self.dRate[self._haps.select(haplotype)] = rate
        self._changed()

    def set_sampling_rate(self, rate, haplotype):
        hs = self._haps.select(haplotype)
        if self._sampling_probability:
            # `rate` is the probability that a removal is a sampling: split the total removal rate accordingly
            P.quantity(rate, 'sampling probability', upper=1)
            removal = self.dRate[hs] + self.sRate[hs]
            self.dRate[hs] = (1 - rate) * removal
            self.sRate[hs] = rate * removal
        else:
            P.quantity(rate, 'sampling rate')
            self.sRate[hs] = rate
        self._changed()

    def set_mutation_rate(self, rate, haplotype, mutation):
        P.quantity(rate, 'mutation rate')
        self._haps.check(haplotype)
        self._sites_axis.check(mutation)
        self.mRate[np.ix_(self._haps.indices(haplotype), self._sites_axis.indices(mutation))] = rate
        self._changed()

    def set_mutation_probabilities(self, probabilities, haplotype, mutation):
        for weight in P.fixed_list(probabilities, 'probabilities list', 4):
            P.quantity(weight, 'mutation probabilities')
        self._haps.check(haplotype)
        self._sites_axis.check(mutation)
        for h in self._haps.indices(haplotype):
            for site in self._sites_axis.indices(mutation):
                # the three OTHER alleles in A, T, C, G order: the haplotype's own allele is left out
                own = self._haps.allele(int(h), int(site))
                others = [w for allele, w in enumerate(probabilities) if allele != own]
                if sum(others) == 0:
                    raise ValueError('Incorrect probabilities list. The sum of three elements without mutation allele should be more 0.')
                self.hapMutType[h, site, :] = others
        self._changed()

    def set_mutation_position(self, mutation, position):
        self._sites_axis_named('number of site').check(mutation, required=True, lists=False)
        P.Axis(self._genome_length, 'mutation position').check(position, required=True, lists=False)
        taken = self.sitesPosition == position
        taken[mutation] = False
        if taken.any():
            raise IndexError("Incorrect value of position. Two mutations can't have the same position.")
        self.sitesPosition[mutation] = position

    def set_susceptibility_type(self, susceptibility_type, haplotype):
        self._groups.check(susceptibility_type, required=True, lists=False)
        self.suscType[self._haps.select(haplotype)] = susceptibility_type
        self._changed()

    def set_susceptibility(self, rate, haplotype, susceptibility_type):
        P.quantity(rate, 'susceptibility rate')
        self._haps.check(haplotype)
        self._groups.check(susceptibility_type)
        self._susceptibility[np.ix_(self._haps.indices(haplotype), self._groups.indices(susceptibility_type))] = rate
        self._changed()

    def set_immunity_transition(self, rate, source, target):
        P.quantity(rate, 'immunity transition rate')
        self._groups.check(source)
        self._groups.check(target)
        block = np.ix_(self._groups.indices(source), self._groups.indices(target))
        keep = np.diagonal(self.suscepTransition).copy()      # a group never "transitions" to itself
        self.suscepTransition[block] = rate
        np.fill_diagonal(self.suscepTransition, keep)
        self._changed()

    def set_population_size(self, amount, population):
        if self.first_simulation:
            raise ValueError('Changing population size is available only before first simulation!')
        P.count(amount, 'population size')
        demes = self._demes.select(population, lists=False)
        self.sizes[demes] = amount
        self._susceptible[demes, :] = 0
        self._susceptible[demes, 0] = amount
        self._changed()

    def _only_before_first_run(self):
        if self.first_simulation:
            raise ValueError('This function is available only before first simulation!')

    def set_susceptible(self, amount, source_type, target_type, population):
        # The reference raises TypeError here unconditionally (it calls check_amount(amount) without the `smth`
        # argument, src/_BirthDeath.pyx:1596, quirk Q11); implemented as documented: move `amount` hosts of every
        # selected deme from one susceptibility group to another.
        self._only_before_first_run()
        P.count(amount, 'amount')
        self._groups.check(source_type, lists=False)
        self._groups.check(target_type, lists=False)
        if source_type == target_type:
            raise ValueError("Source and target susceptibility type shouldn't be equal!")
        for deme in self._demes.select(population):
            if self._susceptible[deme, source_type] < amount:
                raise ValueError('Number of susceptible minus amount should be more or equal 0.')
            if self._susceptible[deme, target_type] + amount > self.sizes[deme]:
                raise ValueError('Number of susceptible plus amount should be equal or less population size.')
            self._susceptible[deme, source_type] -= amount
            self._susceptible[deme, target_type] += amount
        self._changed()

    def set_infectious(self, amount, source_type, target_haplotype, population):
        # see set_susceptible: broken upstream (Q11); implemented as documented.
        self._only_before_first_run()
        P.count(amount, 'amount')
        self._groups.check(source_type, lists=False)
        haps = self._haps.select(target_haplotype, lists=False)
        for deme in self._demes.select(population):
            for h in haps:
                if self._susceptible[deme, source_type] < amount:
                    raise ValueError('Number of susceptible minus amount should be more or equal 0.')
                if self._infectious[deme, h] + amount > self.sizes[deme]:
                    raise ValueError('Number of infectious plus amount should be equal or less population size.')
                self._susceptible[deme, source_type] -= amount
                self._infectious[deme, h] += amount
        self._changed()

    def set_contact_density(self, value, population):
        P.quantity(value, 'contact density')
        demes = self._demes.select(population)
        self.contactDensity[demes] = value
        self.contactDensityBeforeLockdown[demes] = value
        self._cd_touched[demes] = True      # only these demes' LIVE density is overwritten at the next upload
        self._changed()

    def set_npi(self, parameters, population):
        after, start, end = P.fixed_list(parameters, 'npi parameters', 3)
        P.quantity(after, 'first npi parameter')
        P.quantity(start, 'second npi parameter', upper=1)
        P.quantity(end, 'third npi parameter', upper=1)
        demes = self._demes.select(population)
        self.contactDensityAfterLockdown[demes] = after
        self.startLD[demes] = start
        self.endLD[demes] = end
        self._changed()

    def set_sampling_multiplier(self, multiplier, population):
        P.quantity(multiplier, 'sampling multiplier')
        self.samplingMultiplier[self._demes.select(population)] = multiplier
        self._changed()

    def set_migration_probability(self, probability, source, target):
        P.quantity(probability, 'migration probability', upper=1)
        self._demes.check(source)
        self._demes.check(target)
        block = np.ix_(self._demes.indices(source), self._demes.indices(target))
        keep = np.diagonal(self.migrationRates).copy()
        self.migrationRates[block] = probability
        np.fill_diagonal(self.migrationRates, keep)
        P.close_migration_matrix(self.migrationRates)
        self._changed()

    def set_total_migration_probability(self, total_probability):
        P.quantity(total_probability, 'total migration probability', upper=1)
        self.migrationRates[...] = total_probability / (self.popNum - 1)
        np.fill_diagonal(self.migrationRates, 1.0 - total_probability)
        P.close_migration_matrix(self.migrationRates)
        self._changed()

    # ------------------------------------------------------------------ device plumbing
    def param_arrays(self):
        """The parameter block in the order the C ABI (and the test oracle) takes it."""
        c = np.ascontiguousarray
        return dict(b=c(self.bRate), d=c(self.dRate), s=c(self.sRate), mRate=c(self.mRate),
                    hapMutType=c(self.hapMutType), sigma=c(self._susceptibility), suscType=c(self.suscType),
                    T=c(self.suscepTransition), m=c(self.migrationRates), cd=c(self.contactDensity),
                    cdBefore=c(self.contactDensityBeforeLockdown), cdAfter=c(self.contactDensityAfterLockdown),
                    startLD=c(self.startLD), endLD=c(self.endLD), sm=c(self.samplingMultiplier), sizes=c(self.sizes))

    def _ensure_handle(self):
        if self._handle is None:
            self._handle = _capi.Handle(self.sites, self.popNum, self.susNum, self.replicates, 1, self._device)
            seeds = (np.uint64(self.user_seed) + np.arange(self.replicates, dtype=np.uint64)).astype(np.uint64)
            self._handle.set_seeds(seeds)
        return self._handle

    def _sync_params(self):
        if self.recombination > 0:
            raise NotImplementedError(_RECOMB_TEXT)
        h = self._ensure_handle()
        if self._dirty:
            # only demes addressed by set_contact_density since the last upload have their LIVE density overwritten
            # (the reference's setter touches just those, :1633-1640); a deme in lockdown keeps its lockdown density
            h.upload_params(0, self.param_arrays(), reset_contact_density=bool(self._cd_touched.any()),
                            cd_mask=self._cd_touched.astype(np.int32))
            self._cd_touched[:] = False
            self._dirty = False
        if not self.first_simulation:
            R = self.replicates
            h.set_state(np.ascontiguousarray(np.broadcast_to(self._susceptible, (R,) + self._susceptible.shape)),
                        np.ascontiguousarray(np.broadcast_to(self._infectious, (R,) + self._infectious.shape)))
        return h

    def _refresh_host_state(self):
        Sx, I, cd, _ = self._handle.get_state(full=True)
        self._susceptible[...] = Sx[0]
        self._infectious[...] = I[0]
        # CheckLockdown rewrites contactDensity in place (src/_BirthDeath.pyx:698-710): the property shows the live value
        self.contactDensity[...] = cd[0]
        c = self._handle.get_counters()
        self._counters = c

    # ------------------------------------------------------------------ hot path entry points
    def SimulatePopulation(self, iterations, sample_size, time, attempts):
        """Direct (Gillespie) method, reference src/_BirthDeath.pyx:396-429."""
        h = self._sync_params()
        size = self._log_rows() + int(iterations)      # events.size after CreateEvents(iterations)
        h.simulate_direct(int(iterations), int(sample_size), float(time), int(attempts))
        self.first_simulation = True
        self._genealogy_done = False
        self._refresh_host_state()
        self._print_stop_reason(sample_size, time, size)

    def SimulatePopulation_tau(self, iterations, sample_size, time, attempts, leap_block=None):
        """Tau-leaping, reference src/_BirthDeath.pyx:2293-2346.  `leap_block` (not in the reference): run the call in
        blocks of that many leaps and keep finished blocks as a sparse archive instead of dense count rows."""
        h = self._sync_params()
        size = self._log_rows() + int(iterations)
        if leap_block is None:
            h.simulate_tau(int(iterations), int(sample_size), float(time), int(attempts))
        else:
            h.simulate_tau_blocks(int(iterations), int(sample_size), float(time), int(attempts), int(leap_block))
        self.first_simulation = True
        self._genealogy_done = False
        self._refresh_host_state()
        self._print_stop_reason(sample_size, time, size)

    def resample(self, source):
        """Replicate r continues the run of replicate source[r] (source: integers, one per replicate): state, counters,
        logs and lockdown records are copied on the device, the seed and the parameter point stay with r.  A replicate
        that is copied from keeps its own run (source[source[r]] == source[r], what `resample.systematic_map` builds).
        The genealogy is dropped, as after a simulate call."""
        s = np.asarray(source)
        if s.shape != (self.replicates,) or not np.issubdtype(s.dtype, np.integer):
            raise ValueError("resample: source must be an integer array of length %d (got %s of shape %s)"
                             % (self.replicates, s.dtype, s.shape))
        h = self._sync_params()
        h.resample(s)
        self._genealogy_done = False
        self._refresh_host_state()

    def _log_rows(self):
        """events.ptr of replicate 0 before a call (0 before the first one)."""
        c = getattr(self, "_counters", None)
        return int(c['events'][0]) if c is not None and self.first_simulation else 0

    def _print_stop_reason(self, sample_size, time, size):
        """The messages of src/_BirthDeath.pyx:420-429 / :2336-2345 (single-chain use only)."""
        if self.replicates != 1:
            return
        c = self._counters
        if c['globalInfectious'][0] == 0:
            print('Simulation finished because no infections individuals remain!')
        if int(c['events'][0]) >= size:
            print("Achieved maximal number of iterations.")
        if c['sCounter'][0] > sample_size and sample_size != -1:
            print("Achieved sample size.")
        if c['time'][0] > time and time != -1:
            print("Achieved internal time limit.")
        if c['sCounter'][0] <= 1:
            print('\033[41m{}\033[0m'.format('WARNING!'), 'Simulated less 2 samples, so genealogy will not work!')

    def GetGenealogy(self, seed, uniform_stream=None):
        """Backward coalescent replay, reference src/_BirthDeath.pyx:743-1000.

        ``uniform_stream`` (parity tap): per-replicate list of fp64 uniforms consumed in the
        reference's order instead of the device Philox stream.
        """
        if self._handle is None or not self.first_simulation:
            raise RuntimeError('Nothing was simulated. Use simulate() before genealogy().')
        c = self._handle.get_counters()
        if self.replicates == 1 and c['sCounter'][0] < 2:
            print("Less than two cases were sampled...")
            print("_________________________________")
            raise RuntimeError('Less than two cases were sampled.')
        self._handle.genealogy(seed, uniform_stream)
        self._genealogy_done = True
        # the replay rewinds the device infectious counts to the initial state (reference quirk Q9)
        self._refresh_host_state()

    def Stats(self, time_simulation):
        """reference src/_BirthDeath.pyx:2048-2068 (replicate 0; batch runs print aggregate lines)."""
        self.last_elapsed = time_simulation
        c = self._counters
        if self.replicates != 1:
            ev = (c['bCounter'] + c['dCounter'] + c['sCounter'] + c['mCounter'] + c['iCounter'] + c['migPlus']).sum()
            print("Replicates:", self.replicates, " total events:", int(ev), " simulation time:", time_simulation)
            print('----------------------------------')
            return
        print("Number of samples:", int(c['sCounter'][0]))
        print("Total number of iterations:", int(c['events'][0]))
        print('Success number:', int(c['good_attempt'][0]))
        print("Epidemic time:", float(c['time'][0]))
        print('Simulation time:', time_simulation)
        print('Number of infections:', int(c['bCounter'][0]))
        print('Number of recoveries:', int(c['dCounter'][0]))
        if self.sites >= 1:
            print('Number of mutations:', int(c['mCounter'][0]))
        if self.popNum >= 2:
            print('Number of accepted migrations:', int(c['migPlus'][0]))
            print('Number of rejected migrations:', int(c['migNonPlus'][0]))
        if np.any(self.suscepTransition.sum(axis=1) != 0.0):
            print('Number of immunity transitions:', int(c['iCounter'][0]))
        print('----------------------------------')

    # ------------------------------------------------------------------ outputs (reference :1725-1851, 1948-2045)
    def counters(self):
        """Per-replicate counters as a dict of int64 arrays (bCounter ... migNonPlus, events, time)."""
        return self._handle.get_counters()

    def get_chain_events(self, replicate=0):
        """6 x N float64 array in the layout of export_chain_events (src/_BirthDeath.pyx:1849-1851)."""
        return self._handle.get_event_log(replicate)

    def export_chain_events(self, name_file, replicate=0):
        np.save(name_file, self.get_chain_events(replicate))

    def get_multievents(self, replicate=0):
        return self._handle.get_multievents(replicate)

    def export_settings(self, file_template):
        """Writes the model as the command-line tool's parameter files <file_template>/<file_template>.{rt,pp,mg,su,st}
        (reference src/_BirthDeath.pyx:1853-1907; same text, written without changing the working directory) and
        prints the matching command line.  `vgsim_b200.io.read_*` / `python -m vgsim_b200.cli` read them back."""
        import os
        from . import io as _io
        if not os.path.isdir(file_template):
            os.mkdir(file_template)
        base = os.path.join(file_template, os.path.basename(os.path.normpath(file_template)))
        _io.write_settings(base, [self.calculate_string_from_haplotype(h) for h in range(self.hapNum)], self.param_arrays())
        print('Command line command: ' + base + '.rt -pm ' + base + '.pp ' + base + '.mg -su ' + base + '.su -st ' + base + '.st ')

    def set_chain_events(self, name_file, replicate=0):
        """Working counterpart of the reference's set_chain_events (src/_BirthDeath.pyx:1705-1719; upstream it assigns
        to attributes the cdef class does not have).  Loads ``<name_file>.npy`` in the export_chain_events layout
        (direct-method rows; the zero rows the reference saves past its write pointer are dropped), installs it as the
        event log of `replicate` and sets the infectious counts to the state at the end of that log, so that
        genealogy() can replay it.  Epidemic curves need the initial snapshot of a simulate() call and are not defined
        for an imported log."""
        tokens = np.load(name_file + '.npy')
        if tokens.ndim != 2 or tokens.shape[0] != 6:
            raise ValueError('Incorrect chain of events: a 6 x N array is expected.')
        n = int(np.count_nonzero(tokens[0]))            # every real row has time > 0
        chain = np.ascontiguousarray(tokens[:, :n], dtype=np.float64)
        ty, hap, pop, nhap, npop = (chain[k].astype(np.int64) for k in range(1, 6))
        I = self._infectious.astype(np.int64).copy()
        if I.sum() == 0:                                # FirstInfection (:234-242)
            I[0, 0] += 1
        for mask, p, h, v in ((ty == 0, pop, hap, 1), ((ty == 1) | (ty == 2), pop, hap, -1), (ty == 3, pop, hap, -1),
                              (ty == 3, pop, nhap, 1), (ty == 5, npop, hap, 1)):
            np.add.at(I, (p[mask], h[mask]), v)
        if I.min() < 0:
            raise ValueError('Incorrect chain of events: it does not replay from the configured initial state.')
        h = self._sync_params()
        h.set_event_log(replicate, chain, I)
        self.first_simulation = True
        self._genealogy_done = False
        self._refresh_host_state()

    def _require_tree(self):
        if not self._genealogy_done:
            print('Genealogy was not simulated. Use VGsim.genealogy() method to simulate it.')
            raise RuntimeError('Genealogy was not simulated.')

    def get_tree(self, replicate=0):
        self._require_tree()
        tree, pop, times = self._handle.get_tree(replicate)
        return tree, times

    def get_tree_populations(self, replicate=0):
        self._require_tree()
        return self._handle.get_tree(replicate)[1]

    def get_mutations(self, replicate=0):
        """(nodeId, AS, DS, site, time) arrays, src/models.pxi:12-26."""
        self._require_tree()
        return self._handle.get_mutations(replicate)

    def get_migrations(self, replicate=0):
        """(nodeId, time, oldPop, newPop) arrays, src/models.pxi:42-46."""
        self._require_tree()
        return self._handle.get_migrations(replicate)

    def export_ts_tables(self, replicate=0):
        """The rows the reference's export_ts (src/_BirthDeath.pyx:1909-1946) hands to a tskit.TableCollection, as numpy
        columns in the order it adds them (before `tc.sort()`): works without tskit, `export_ts` feeds them to it.
        Times are tskit times: `times[0] - t` (time before the node 0, the reference's convention)."""
        self._require_tree()
        tree, pop, times = self._handle.get_tree(replicate)
        n_nodes = len(tree)
        L = float(self._genome_length)
        t0 = times[0] if n_nodes else 0.0
        child = np.arange(max(n_nodes - 1, 0), dtype=np.int64)               # rows 0 .. 2n-3: every node but the last
        is_parent = np.zeros(n_nodes, bool)
        is_parent[tree[child]] = True                                        # child_or_parent[self.tree[i]] = 0
        node, AS, DS, site, mt = self._handle.get_mutations(replicate)
        gnode, gt, gold, gnew = self._handle.get_migrations(replicate)
        pos = self.sitesPosition.astype(np.float64)
        pos = np.where(pos == 0, pos + 1, np.where(pos == L, pos - 1, pos))  # sites must lie strictly inside (0, L)
        allele = np.array(['A', 'T', 'C', 'G'])
        return {
            "sequence_length": L,
            "populations": self.popNum,
            "migrations": {"left": np.zeros(len(gnode)), "right": np.ones(len(gnode)), "node": gnode.astype(np.int64),
                           "source": gold.astype(np.int64), "dest": gnew.astype(np.int64), "time": t0 - gt},
            "edges": {"left": np.zeros(len(child)), "right": np.full(len(child), L), "parent": tree[child].astype(np.int64),
                      "child": child},
            "nodes": {"flags": (~is_parent).astype(np.uint32), "time": t0 - times, "population": pop.astype(np.int64)},
            "sites": {"position": pos, "ancestral_state": np.full(self.sites, 'A')},
            "mutations": {"site": site.astype(np.int64), "node": node.astype(np.int64), "derived_state": allele[DS],
                          "time": t0 - mt},
        }

    def export_ts(self, replicate=0):
        """tskit.TreeSequence of one replicate's genealogy (reference src/_BirthDeath.pyx:1909-1946).  tskit is an
        optional dependency here: without it use export_ts_tables()."""
        try:
            import tskit
            tskit.TableCollection
        except (ImportError, AttributeError) as e:
            raise ImportError("export_ts needs tskit; export_ts_tables() returns the same rows as numpy columns") from e
        tb = self.export_ts_tables(replicate)
        tc = tskit.TableCollection()
        tc.sequence_length = tb["sequence_length"]
        m = tb["migrations"]
        for i in range(len(m["node"])):
            tc.migrations.add_row(m["left"][i], m["right"][i], int(m["node"][i]), int(m["source"][i]), int(m["dest"][i]),
                                  float(m["time"][i]))
        for _ in range(tb["populations"]):
            tc.populations.add_row(None)
        e_ = tb["edges"]
        for i in range(len(e_["child"])):
            tc.edges.add_row(e_["left"][i], e_["right"][i], int(e_["parent"][i]), int(e_["child"][i]))
        nd = tb["nodes"]
        for i in range(len(nd["time"])):
            tc.nodes.add_row(int(nd["flags"][i]), float(nd["time"][i]), int(nd["population"][i]))
        st = tb["sites"]
        for i in range(len(st["position"])):
            tc.sites.add_row(float(st["position"][i]), str(st["ancestral_state"][i]))
        mu = tb["mutations"]
        for i in range(len(mu["node"])):
            tc.mutations.add_row(site=int(mu["site"][i]), node=int(mu["node"][i]), derived_state=str(mu["derived_state"][i]),
                                 time=float(mu["time"][i]))
        tc.sort()
        return tc.tree_sequence()

    def print_mutations(self, replicate=0):
        """Reference src/_BirthDeath.pyx:1176-1179: one tuple (nodeId, DS, AS, site, time) per line."""
        self._require_tree()
        node, AS, DS, site, t = self._handle.get_mutations(replicate)
        print('nodeId\tDS\tAS\tsite\ttime')
        for i in range(len(node)):
            print((int(node[i]), int(DS[i]), int(AS[i]), int(site[i]), float(t[i])))

    def print_migrations(self, replicate=0):
        """Reference src/_BirthDeath.pyx:1181-1184: one tuple (nodeId, time, oldPop, newPop) per line."""
        self._require_tree()
        node, t, oldp, newp = self._handle.get_migrations(replicate)
        print('nodeId\ttime\tsource population\ttarget population')
        for i in range(len(node)):
            print((int(node[i]), float(t[i]), int(oldp[i]), int(newp[i])))

    def output_tree_mutations(self, replicate=0):
        self._require_tree()
        tree, pop, times = self._handle.get_tree(replicate)
        node, AS, DS, site, t = self._handle.get_mutations(replicate)
        mut = [list(map(int, node)), list(map(int, AS)), list(map(int, site)), list(map(int, DS)), list(map(float, t))]
        # The reference maps node -> deme through a {time: events.populations} dict, which is garbage
        # for tau-phase nodes (quirk Q14); the replacement keys the same dict by node time but fills it
        # from tree_pop, which is what the dict was meant to hold.
        populations = {float(times[i]): int(pop[i]) for i in range(len(times))}
        return tree, times, mut, populations

    def export_migrations(self, name_file, file_path, replicate=0):
        self._require_tree()
        node, t, oldp, newp = self._handle.get_migrations(replicate)
        from . import io as _io
        fn = (file_path + '/' if file_path is not None else '') + name_file + '.tsv'
        with open(fn, 'w') as f:
            f.writelines(_io.migration_lines(node, t, oldp, newp))

    def output_sample_data(self, replicate=0):
        ev = self.get_chain_events(replicate)
        sel = ev[1] == SAMPLING
        return list(ev[0][sel]), [int(x) for x in ev[3][sel]], [int(x) for x in ev[2][sel]]

    # ---- epidemic curves (reference :1967-2045), computed for every compartment in one device pass over the log
    def epidemic_curves(self, step_num, rep_first=0, rep_count=None,
                        want=("infectious", "susceptible", "removed", "sampled")):
        """True compartment counts on the reference's time grid for a range of replicates (see
        include/vgsim_b200.h: vgsim_epidemic_curves)."""
        return self._handle.epidemic_curves(step_num, rep_first, rep_count, want)

    def trajectories(self, times):
        """Every replicate's epidemic on one time grid shared by all replicates, from one device pass over each log.

        `times`: absolute times, finite and strictly increasing.  Returns a dict of int64 arrays ``infectious_deme``
        [R, T, K], ``infectious_hap`` [R, T, H], ``sampled_deme`` [R, T, K] and ``sampled_hap`` [R, T, H]: the state after
        every log row with time <= times[j], samplings counted from the start of the log.  A point after a replicate's
        current time was not simulated for it: every entry of that replicate's row at that point is -1."""
        if self._handle is None:
            raise RuntimeError('Nothing was simulated. Use simulate() before trajectories().')
        return self._handle.trajectories(times)

    def lineages_through_time(self, times):
        """int64 [R, T]: the lineages of each replicate's genealogy alive at times[j] (nodes with time >= times[j] whose
        parent is older than times[j], or that are roots), times absolute like get_tree's; zeros for a replicate
        without a tree.  Needs genealogy() after the last simulate()."""
        self._require_tree()
        return self._handle.lineages_through_time(times)

    def _lockdown_rows(self, pop, replicate):
        state, lp, lt = self._handle.get_lockdowns(replicate)
        return [[int(state[i]), float(lt[i])] for i in range(len(state)) if int(lp[i]) == pop]

    def _tau_migration_in(self, pop, replicate):
        """Per leap: counts[leap][S][H] of MIGRATION multi-events into deme `pop`, and the leap times."""
        K, H, S = self.popNum, self.hapNum, self.susNum
        counts, tt = self._handle.get_tau_log(replicate)
        if counts.shape[0] == 0 or K < 2:
            return np.zeros((0, S, H), np.int64), np.zeros(0)
        mig = counts[:, :K * (K - 1) * S * H].reshape(-1, K, K - 1, S, H).astype(np.int64)  # [leap][source][target'][s][h]
        tot = np.zeros((counts.shape[0], S, H), np.int64)
        for sp in range(K):
            if sp != pop:
                tot += mig[:, sp, pop - (1 if pop > sp else 0)]
        return tot, tt[:, 0]

    def get_data_infectious(self, pop, hap, step_num, replicate=0):
        """(Data, Sample, time_points, Lockdowns) exactly as the reference returns them (:1967-2005).  Its DEATH /
        SAMPLING branch reads `DEATH or SAMPLING or MUTATION and <this cell>`, so EVERY recovery and sampling of the
        replicate is subtracted from Data and every sampling is counted in Sample, and grid points after the one
        holding the last log row stay zero; both are rebuilt here from the true counts of `epidemic_curves`."""
        c = self._handle.epidemic_curves(step_num, replicate, 1, ("infectious", "removed", "sampled"))
        last = int(c["last_point"][0])
        removed_all = c["removed"][0].sum(axis=(1, 2))
        Data = (c["infectious"][0, :, pop, hap] + c["removed"][0, :, pop, hap] - removed_all).astype(np.float64)
        Sample = c["sampled"][0].sum(axis=(1, 2)).astype(np.float64)
        Data[last + 1:] = 0.0
        Sample[last + 1:] = 0.0
        return Data, Sample, [float(x) for x in c["time_points"][0]], self._lockdown_rows(pop, replicate)

    def get_data_susceptible(self, pop, sus, step_num, replicate=0):
        """(Data, time_points, Lockdowns) exactly as the reference returns them (:2008-2045).  Direct-method rows give
        the true count; for MULTITYPE rows the reference matches MIGRATION records on `haplotypes == sus` instead of
        `newHaplotypes == sus` (:2037): that difference is rebuilt from the migration block of the dense tau log."""
        c = self._handle.epidemic_curves(step_num, replicate, 1, ("susceptible",))
        last = int(c["last_point"][0])
        tp = c["time_points"][0]
        Data = c["susceptible"][0, :, pop, sus].astype(np.float64)
        mig, lt = self._tau_migration_in(pop, replicate)
        if mig.shape[0]:
            by_group = mig[:, sus, :].sum(axis=1)
            by_hap = mig[:, :, sus].sum(axis=1) if sus < self.hapNum else np.zeros(len(lt), np.int64)
            # a leap lands on the first grid point that is not before it (:2016-2018), capped at the last point
            pt = np.minimum(np.searchsorted(tp, lt, side="left"), step_num)
            corr = np.zeros(step_num + 1)
            np.add.at(corr, pt, (by_group - by_hap).astype(np.float64))
            Data += np.cumsum(corr)
        Data[last + 1:] = 0.0
        return Data, [float(x) for x in tp], self._lockdown_rows(pop, replicate)

    def output_epidemiology_timelines(self, step_num, output_file, replicate=0):
        """Reference src/_BirthDeath.pyx:1765-1847 (semantics and quirks in vgsim_b200/io.py: epidemiology_timelines)."""
        from . import io as _io
        c = self._handle.get_counters()
        times, sus, inf = _io.epidemiology_timelines(self.get_chain_events(replicate), self.sizes, self.popNum, self.susNum,
                                                     self.hapNum, float(c["time"][replicate]), int(step_num))
        if output_file == True:  # noqa: E712  (the reference compares with == True)
            _io.write_timelines(times, sus, inf)
            return None
        return _io.timelines_as_dict(times, sus, inf)

    def get_lockdowns(self, replicate=0):
        return self._handle.get_lockdowns(replicate)

    def PrintCounters(self):
        c = self._counters
        print("Birth counter(mutable): ", int(c['bCounter'][0]))
        print("Death counter(mutable): ", int(c['dCounter'][0]))
        print("Sampling counter(mutable): ", int(c['sCounter'][0]))
        print("Mutation counter(mutable): ", int(c['mCounter'][0]))
        print("Immunity transition counter(mutable):", int(c['iCounter'][0]))
        print("Migration counter(mutable):", int(c['migPlus'][0]))

    def get_proportion(self):
        c = self._counters
        return int(c['migNonPlus'][0]) / (int(c['events'][0]) - 1)

    def propensities(self, replicate=0):
        """Deterministic parity tap (PrintPropensities, src/_BirthDeath.pyx:2615-2649): the P tau-leap
        propensities of the current state in positional channel order, plus drifts and tau."""
        h = self._sync_params()
        return h.propensities(replicate)

    def PrintPropensities(self):
        prop, dI, dS, tau = self.propensities()
        K, H, S, U = self.popNum, self.hapNum, self.susNum, self.sites
        k = 0
        print("Migrations")
        for s in range(K):
            for r in range(K):
                if s == r:
                    continue
                for i in range(S):
                    for h in range(H):
                        print(s, r, i, h, prop[k]); k += 1
        for s in range(K):
            print("Susceptibility transition")
            for i in range(S):
                for j in range(S):
                    if i == j:
                        continue
                    print(s, i, j, prop[k]); k += 1
            for h in range(H):
                print("Recovery ", s, h, self.suscType[h], prop[k]); k += 1
                print("Sampling ", s, h, self.suscType[h], prop[k]); k += 1
                for site in range(U):
                    for i in range(3):
                        print("Mutation", s, h, site, i, prop[k]); k += 1
                for i in range(S):
                    print("Transmission", s, h, i, prop[k]); k += 1

    def rates(self, replicate=0):
        """Deterministic parity tap for the direct method (UpdateAllRates, src/_BirthDeath.pyx:279-351)."""
        h = self._sync_params()
        return h.rates(replicate)
