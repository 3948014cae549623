"""`Simulator` — the public API of the reference (src/_interface.py:9-883), kept signature-compatible.

Every method delegates to ``self.simulation`` exactly like the reference wrapper does; what changed is
what ``self.simulation`` is (``vgsim_b200._engine.BirthDeathModel``: plain-Python parameter store over
the sm_100a kernels).  Plotting (matplotlib) and the reference's interface methods that call engine
methods which do not exist upstream (SURVEY quirk Q12) are out of scope and raise NotImplementedError.

Extension: ``replicates=R`` simulates R independent replicates (seed + r) in one batched launch.
"""
import sys
import time
from random import randrange

import numpy as np

from ._engine import BirthDeathModel
from .io import writeGenomeNewick, writeMutations


class Simulator:
    def __init__(self, number_of_sites=0, populations_number=1, number_of_susceptible_groups=1, seed=None,
                 sampling_probability=False, memory_optimization=False, genome_length=int(1e6),
                 recombination_probability=0.0, replicates=1, device=None, verbose=True):
        self.fig = None
        self.verbose = verbose
        if seed == None:
            seed = int(randrange(sys.maxsize))
        if verbose:
            print('User seed:', seed)
        self.simulation = BirthDeathModel(number_of_sites=number_of_sites, populations_number=populations_number,
                                          number_of_susceptible_groups=number_of_susceptible_groups, seed=seed,
                                          sampling_probability=sampling_probability,
                                          memory_optimization=memory_optimization, genome_length=genome_length,
                                          recombination_probability=recombination_probability,
                                          replicates=replicates, device=device)

    # ------------------------------------------------------------------ read-only properties
    @property
    def seed(self):
        return self.simulation.seed

    @property
    def sampling_probability(self):
        return self.simulation.sampling_probability

    @property
    def memory_optimization(self):
        return self.simulation.memory_optimization

    @property
    def number_of_sites(self):
        return self.simulation.number_of_sites

    @property
    def haplotypes_number(self):
        return self.simulation.haplotypes_number

    @property
    def populations_number(self):
        return self.simulation.populations_number

    @property
    def number_of_susceptible_groups(self):
        return self.simulation.number_of_susceptible_groups

    @property
    def replicates(self):
        return self.simulation.replicates

    def get_indexes_from_haplotype(self, haplotype):
        return np.array(self.simulation.create_list_for_cycles(haplotype, self.simulation.haplotype_number))

    # ------------------------------------------------------------------ parameters (src/_interface.py:158-473)
    @property
    def initial_haplotype(self):
        return self.simulation.initial_haplotype

    def set_initial_haplotype(self, amount):
        self.simulation.set_initial_haplotype(amount)

    @property
    def step_haplotype(self):
        return self.simulation.step_haplotype

    def set_step_haplotype(self, amount):
        self.simulation.set_step_haplotype(amount)

    @property
    def genome_length(self):
        return self.simulation.genome_length

    def set_genome_length(self, genome_length):
        self.simulation.set_genome_length(genome_length)

    @property
    def coinfection_parameters(self):
        return self.simulation.coinfection_parameters

    def set_coinfection_parameters(self, recombination):
        self.simulation.set_coinfection_parameters(recombination)

    @property
    def transmission_rate(self):
        return self.simulation.transmission_rate

    def set_transmission_rate(self, rate, haplotype=None):
        self.simulation.set_transmission_rate(rate, haplotype)

    @property
    def recovery_rate(self):
        return self.simulation.recovery_rate

    def set_recovery_rate(self, rate, haplotype=None):
        self.simulation.set_recovery_rate(rate, haplotype)

    @property
    def sampling_rate(self):
        return self.simulation.sampling_rate

    def set_sampling_rate(self, rate, haplotype=None):
        self.simulation.set_sampling_rate(rate, haplotype)

    @property
    def mutation_rate(self):
        return self.simulation.mutation_rate

    def set_mutation_rate(self, rate, haplotype=None, mutation=None):
        self.simulation.set_mutation_rate(rate, haplotype, mutation)

    @property
    def mutation_probabilities(self):
        return self.simulation.mutation_probabilities

    def set_mutation_probabilities(self, probabilities, haplotype=None, mutation=None):
        self.simulation.set_mutation_probabilities(probabilities, haplotype, mutation)

    @property
    def mutation_position(self):
        return self.simulation.mutation_position

    def set_mutation_position(self, mutation, position):
        self.simulation.set_mutation_position(mutation, position)

    @property
    def susceptibility_type(self):
        return self.simulation.susceptibility_type

    def set_susceptibility_type(self, susceptibility_type, haplotype=None):
        self.simulation.set_susceptibility_type(susceptibility_type, haplotype)

    @property
    def susceptibility(self):
        return self.simulation.susceptibility

    def set_susceptibility(self, rate, haplotype=None, susceptibility_type=None):
        self.simulation.set_susceptibility(rate, haplotype, susceptibility_type)

    @property
    def immunity_transition(self):
        return self.simulation.immunity_transition

    def set_immunity_transition(self, rate, source=None, target=None):
        self.simulation.set_immunity_transition(rate, source, target)

    @property
    def population_size(self):
        return self.simulation.population_size

    def set_population_size(self, size, population=None):
        self.simulation.set_population_size(size, population)

    @property
    def contact_density(self):
        return self.simulation.contact_density

    def set_contact_density(self, value, population=None):
        self.simulation.set_contact_density(value, population)

    @property
    def npi(self):
        return self.simulation.npi

    def set_npi(self, parameters, population=None):
        self.simulation.set_npi(parameters, population)

    @property
    def sampling_multiplier(self):
        return self.simulation.sampling_multiplier

    def set_sampling_multiplier(self, multiplier, population=None):
        self.simulation.set_sampling_multiplier(multiplier, population)

    @property
    def migration_probability(self):
        return self.simulation.migration_probability

    def set_migration_probability(self, probability, source=None, target=None):
        self.simulation.set_migration_probability(probability, source, target)

    def set_total_migration_probability(self, total_probability):
        self.simulation.set_total_migration_probability(total_probability)

    @property
    def susceptible(self):
        return self.simulation.susceptible

    def set_susceptible(self, amount, source_type, target_type, population=None):
        self.simulation.set_susceptible(amount, source_type, target_type, population)

    @property
    def infectious(self):
        return self.simulation.infectious

    def set_infectious(self, amount, source_type, target_haplotype, population=None):
        self.simulation.set_infectious(amount, source_type, target_haplotype, population)

    # ------------------------------------------------------------------ hot path (src/_interface.py:799-840)
    def simulate(self, iterations=1000, sample_size=None, epidemic_time=-1, method='direct', attempts=200):
        if sample_size is None:
            sample_size = iterations
        if epidemic_time is None:
            epidemic_time = -1
        start_time = time.time()
        if method == 'direct':
            self.simulation.SimulatePopulation(iterations, sample_size, epidemic_time, attempts)
        elif method == 'tau':
            self.simulation.SimulatePopulation_tau(iterations, sample_size, epidemic_time, attempts)
        else:
            print("Unknown method. Choose between 'direct' and 'tau'.")
            return
        if self.verbose:
            self.simulation.Stats(time.time() - start_time)

    def resample(self, source):
        """Replicate r continues the run of replicate source[r], its whole history included; seeds and parameters stay
        with r.  A replicate that is copied from keeps its own run: build maps with `vgsim_b200.resample.systematic_map`
        (resampling by weights) or fork one replicate into all (``[s] * replicates``)."""
        self.simulation.resample(source)

    def genealogy(self, seed=None):
        start_time = time.time()
        self.simulation.GetGenealogy(seed)
        if self.verbose:
            print(f"Getting genealogy time: {time.time() - start_time}")

    # ------------------------------------------------------------------ outputs (src/_interface.py:498-598)
    def export_newick(self, file_template=None, file_path=None, replicate=0):
        pruferSeq, times, mut, populations = self.simulation.output_tree_mutations(replicate)
        pops = self.simulation.get_tree_populations(replicate)
        writeGenomeNewick(pruferSeq, times, pops, file_template, file_path)

    def export_mutations(self, file_template=None, file_path=None, replicate=0):
        pruferSeq, times, mut, populations = self.simulation.output_tree_mutations(replicate)
        writeMutations(mut, len(pruferSeq), file_template, file_path)

    def export_migrations(self, file_template=None, file_path=None, replicate=0):
        self.simulation.export_migrations(file_template, file_path, replicate)

    # the tutorial / notebook spelling (docs "Tutorials and examples", BASELINE north_star)
    output_newick = export_newick
    output_mutations = export_mutations
    output_migrations = export_migrations

    def output_sample_data(self, output_print=False, replicate=0):
        time_, pop, hap = self.simulation.output_sample_data(replicate)
        if output_print:
            return time_, pop, hap
        print(time_)
        print(pop)
        print(hap)

    def export_chain_events(self, file_name="chain_events", replicate=0):
        self.simulation.export_chain_events(file_name, replicate)

    def get_chain_events(self, replicate=0):
        return self.simulation.get_chain_events(replicate)

    def export_settings(self, file_template="parameters"):
        """Exports the model as text parameter files (reference src/_interface.py:578-585)."""
        self.simulation.export_settings(file_template)

    def set_chain_events(self, file_name="chain_events", replicate=0):
        """Imports an event chain saved by export_chain_events (reference src/_interface.py: set_chain_events)."""
        self.simulation.set_chain_events(file_name, replicate)

    def get_data_susceptible(self, population, susceptibility_type, step_num, replicate=0):
        """susceptible, time_points, lockdowns (reference src/_interface.py:599-615)."""
        return self.simulation.get_data_susceptible(population, susceptibility_type, step_num, replicate)

    def get_data_infectious(self, population, haplotype, step_num, replicate=0):
        """infections, sample, time_points, lockdowns (reference src/_interface.py:617-633)."""
        return self.simulation.get_data_infectious(population, haplotype, step_num, replicate)

    def output_epidemiology_timelines(self, step=1000, output_file=False, replicate=0):
        """Compartment counts of every deme over `step` grid intervals (reference src/_interface.py:553-566)."""
        return self.simulation.output_epidemiology_timelines(step, output_file, replicate)

    def epidemic_curves(self, step_num, rep_first=0, rep_count=None):
        """Every compartment of a range of replicates on the reference's time grid, one device pass over the logs."""
        return self.simulation.epidemic_curves(step_num, rep_first, rep_count)

    def trajectories(self, times):
        """Infectious and cumulative sampled counts per deme and per haplotype of every replicate at the absolute times
        `times` (finite, strictly increasing), one grid for all replicates: dict of int64 arrays infectious_deme
        [R, T, K], infectious_hap [R, T, H], sampled_deme [R, T, K], sampled_hap [R, T, H].  A point after a replicate's
        current time was not simulated for it, and every entry of its row there is -1."""
        return self.simulation.trajectories(times)

    def lineages_through_time(self, times):
        """Lineages of each replicate's genealogy alive at the absolute times `times`, int64 [R, T] (after genealogy();
        zeros for a replicate without a tree)."""
        return self.simulation.lineages_through_time(times)

    def get_tree(self, replicate=0):
        return self.simulation.get_tree(replicate)

    def counters(self):
        return self.simulation.counters()

    def get_proportion(self):
        return self.simulation.get_proportion()

    def print_mutations(self, replicate=0):
        self.simulation.print_mutations(replicate)

    def print_migrations(self, replicate=0):
        self.simulation.print_migrations(replicate)

    def print_counters(self):
        self.simulation.PrintCounters()

    def print_propensities(self):
        self.simulation.PrintPropensities()

    def citation(self):
        print("VGsim: scalable viral genealogy simulator for global pandemic")
        print("Vladimir Shchur, Vadim Spirin, Dmitry Sirotkin, EvgeniBurovski, Nicola De Maio, Russell Corbett-Detig")
        print("medRxiv 2021.04.21.21255891; doi: https://doi.org/10.1101/2021.04.21.21255891")

    def export_ts(self, replicate=0):
        """tskit tree sequence of the genealogy (src/_interface.py:593); needs tskit, see export_ts_tables."""
        return self.simulation.export_ts(replicate)

    def export_ts_tables(self, replicate=0):
        """The table rows of export_ts as numpy columns (no tskit needed)."""
        return self.simulation.export_ts_tables(replicate)

    # ------------------------------------------------------------------ out of scope (SURVEY §2: plotting, printing)
    def _out_of_scope(self, *a, **k):
        raise NotImplementedError("outside the hot-path scope of vgsim_b200 (plotting / pretty-printing)")

    add_plot_infectious = add_plot_susceptible = add_legend = add_title = plot = _out_of_scope
    print_basic_parameters = print_populations = print_immunity_model = print_all = _out_of_scope
    export_state = set_settings = set_state = debug = _out_of_scope
    # print_chain / print_tree / print_recomb delegate to engine methods that do not exist upstream either
    plot_infectious = print_chain = print_tree = print_recomb = _out_of_scope
