"""Per-mutant scoring of the reference (utils/energy_scores.py:31-488) on the B200 engine.

`score_sequence(seq, input_file, sim_options) -> ScoreSeq`, `get_mfe_e_ss`, `ScoreSeq` and
`get_first_suboptimal_structure_and_energy` keep the reference's names, arguments and return values.
New here: `score_sequences(seqs, input_file, sim_options)`, the batched form the lock-step replica
loop uses -- ONE engine call (MFE + backtrack + partition function + eval of the target and of every
alternative structure) for all mutants of a Monte-Carlo sub-step, one more for their self-dimers in
avoid mode (`-o on`), then the reference's double-precision score arithmetic on float32-rounded energies
(SURVEY.md 8b "Derived-score arithmetic").

Quirks kept for score parity (SURVEY.md App. C): only the scoring terms present in `sim_options.scoring_f`
are evaluated (the reference's option parser keeps the first `-sf` term only, stats_inputs_outputs.py:232-237,
which is the caller's business, not ours); `fc.mfe()`'s energy is dropped and 'Ed-MFE' folds again (:350-354);
'&' becomes "Ee" for the similarity scores (:79); 1-MCC / 1-precision / 1-recall are stored as complements (:308-333).
"""
from .. import RNA
from . import dimer_multichain_energy as dme
from .sim_score import SimScore

md = RNA.md()
md.compute_bpp = 0

_PK_BRACKETS = ("[]", "<>", "{}")


def get_pk_struct(seq, ss_nopk, fc):
    """Pseudoknot overlay (utils/sequence_utils.py:1166-1228): forbid the positions already paired, fold again,
    paint the new pairs with the next bracket family; up to three rounds, a round runs only while the previous
    one still found pairs.  Hard constraints accumulate on `fc` exactly as in the reference."""
    ss_pk = ss_nopk
    for opn, cls in _PK_BRACKETS:
        constraints = "".join("." if ch == "." else "x" for ch in ss_pk)
        fc.hc_add_from_db(constraints)
        mfe_structure, _ = fc.mfe()
        chars = list(ss_pk)
        for i, ch in enumerate(mfe_structure):
            if ch == "(":
                chars[i] = opn
            elif ch == ")":
                chars[i] = cls
        ss_pk = "".join(chars)
        if "(" not in mfe_structure:
            break
    return ss_pk


def get_pk_structs(structures, compounds):
    """get_pk_struct for all mutants of a sub-step at once: every round is ONE engine call (the constrained refolds of the
    sequences whose previous round still found pairs).  Same result, sequence by sequence, as get_pk_struct."""
    ss_pk = list(structures)
    live = list(range(len(ss_pk)))
    for opn, cls in _PK_BRACKETS:
        if not live:
            break
        for k in live:
            compounds[k].hc_add_from_db("".join("." if ch == "." else "x" for ch in ss_pk[k]))
        RNA.fold_compound.prefetch_constrained([compounds[k] for k in live])
        still = []
        for k in live:
            mfe_structure, _ = compounds[k].mfe()
            chars = list(ss_pk[k])
            for i, ch in enumerate(mfe_structure):
                if ch == "(":
                    chars[i] = opn
                elif ch == ")":
                    chars[i] = cls
            ss_pk[k] = "".join(chars)
            if "(" in mfe_structure:
                still.append(k)
        live = still
    return ss_pk


def get_mfe_e_ss(seq, sim_options):
    """(Epf, MFE structure, fold compound) -- energy_scores.py:128-159.  Single chain: ensemble free energy from
    fc.pf(), structure from fc.mfe() (+ pseudoknot overlay when sim_options.pks == "on"); two chains: structure from
    fc.mfe_dimer() with '&' re-inserted after strand A, energy = FAB = fc.pf_dimer()[-1]."""
    fc = RNA.fold_compound(seq, md)
    if sim_options.oligo_state in {"none", "avoid"}:
        _, energy = fc.pf()
        structure = fc.mfe()[0]
        if sim_options.pks == "on":
            structure = get_pk_struct(seq, structure, fc)
    elif sim_options.oligo_state in {"homodimer", "heterodimer"}:
        seqa_len = len(seq.split("&")[0])
        structure_dim = fc.mfe_dimer()[0]
        energy = fc.pf_dimer()[-1]
        structure = structure_dim[:seqa_len] + "&" + structure_dim[seqa_len:]
    else:
        raise ValueError("unknown oligo_state: %r" % (sim_options.oligo_state,))
    return energy, structure, fc


def _score_with_compound(seq, input_file, sim_options, pf_energy, mfe_structure, fold_comp, dimer_comp=None):
    s = ScoreSeq(sequence=seq)
    s.get_Epf(pf_energy)
    s.get_mfe_ss(mfe_structure)
    s.get_edesired(fold_comp.eval_structure(input_file.sec_struct.replace("&", "")))
    s.get_edesired_minus_Epf(s.Epf, s.edesired)

    ssc = SimScore(input_file.sec_struct.replace("&", "Ee"), s.mfe_ss.replace("&", "Ee"))
    ssc.find_basepairs()
    ssc.cofusion_matrix()
    s.get_precision(ssc.precision())
    s.get_recall(ssc.recall())
    s.get_mcc(ssc.mcc())

    for function, weight in sim_options.scoring_f:
        if function == "sln_Epf":
            s.get_sln_Epf()
        if function == "Ed-MFE":
            s.get_MFE()
            s.get_edesired_minus_MFE()
        if function == "Edef":
            s.get_ensemble_defect(input_file.sec_struct)
    s.get_scoring_function(sim_options.scoring_f)

    if input_file.alt_sec_struct is not None:
        energies = [fold_comp.eval_structure(alt_dbn) for alt_dbn in input_file.alt_sec_structs]
        s.get_edesired2(sum(energies) / len(energies))
        s.get_edesired2_minus_Epf(s.Epf, s.edesired2)
        s.get_scoring_function_w_alt_ss()

    if sim_options.subopt == "on" and s.mcc == 0:
        s.get_subopt_e(get_first_suboptimal_energy(seq, fold_comp))
        s.get_esubopt_minus_Epf(s.Epf, s.subopt_e)
        s.get_scoring_function_w_subopt()

    if sim_options.oligo_state in ("heterodimer", "homodimer"):
        halves = input_file.sec_struct.split("&")
        if sim_options.oligo_state == "heterodimer" or halves[0] != halves[1]:
            s.get_scoring_function_oligomer(fold_comp)
        else:
            s.get_scoring_function_homomonomer(fold_comp)
    if sim_options.oligo_state == "avoid":
        s.get_scoring_function_monomer(dimer_comp)

    if sim_options.motifs:
        s.update_scoring_function_w_motifs(score_motifs(seq, sim_options))
    return s


def score_motifs(seq, sim_options):
    """utils/sequence_utils.py:1231-1256: sum of the bonuses of the motifs (compiled regex, weight) found in seq"""
    total = 0
    for motif in sim_options.motifs:
        if sim_options.motifs[motif][0].search(seq):
            total += sim_options.motifs[motif][1]
    return total


def score_sequence(seq, input_file, sim_options):
    """energy_scores.py:31-125, one sequence (three small engine calls).  Prefer score_sequences() in loops."""
    pf_energy, mfe_structure, fold_comp = get_mfe_e_ss(seq, sim_options)
    return _score_with_compound(seq, input_file, sim_options, pf_energy, mfe_structure, fold_comp)


def score_sequences(seqs, input_file, sim_options):
    """Batched score_sequence: one engine call for the fold + eval work of all `seqs` (the R mutants of one
    Monte-Carlo sub-step, energy_scores.py:70-99), then the per-sequence bookkeeping.  Returns a list of ScoreSeq
    equal, field by field, to [score_sequence(s, ...) for s in seqs]."""
    seqs = list(seqs)
    if not seqs:
        return []
    compounds = [RNA.fold_compound(s, md) for s in seqs]
    targets = [input_file.sec_struct]
    if input_file.alt_sec_struct is not None:
        targets += list(input_file.alt_sec_structs)
    targets = [t.replace("&", "") for t in targets]
    RNA.fold_compound.prefetch(compounds, [targets] * len(seqs))
    dimer = sim_options.oligo_state in {"homodimer", "heterodimer"}
    folded = []
    for seq, fc in zip(seqs, compounds):
        if dimer:
            a = len(seq.split("&")[0])
            sd = fc.mfe_dimer()[0]
            folded.append((fc.pf_dimer()[-1], sd[:a] + "&" + sd[a:]))
        else:
            folded.append((fc.pf()[1], fc.mfe()[0]))
    structures = [f[1] for f in folded]
    if not dimer and sim_options.pks == "on":
        structures = get_pk_structs(structures, compounds)
    dimers = [None] * len(seqs)
    if sim_options.oligo_state == "avoid":
        # the self-dimers seq&seq of all mutants in one more engine call: partition function only, as get_scoring_function_monomer
        # asks of each on its own
        dimers = [RNA.fold_compound(s + "&" + s) for s in seqs]
        RNA.fold_compound.prefetch(dimers, want=RNA._eng.WANT_PF)
    return [_score_with_compound(seq, input_file, sim_options, f[0], ss, fc, dc)
            for seq, f, ss, fc, dc in zip(seqs, folded, structures, compounds, dimers)]


class ScoreSeq:
    """Score record of one sequence; field and method names are the reference's (energy_scores.py:162-450)
    because DesiRNA.py:373-375 dumps vars(ScoreSeq) into its trajectory files."""

    def __init__(self, sequence):
        self.sequence = sequence
        self.scoring_function = 0
        self.replica_num = None
        self.temp_shelf = None
        self.sim_step = 0
        self.edesired_minus_Epf = 0
        self.Epf = 0
        self.edesired = 0
        self.mcc = 0
        self.mcc_alt = 0
        self.mfe_ss = None
        self.subopt_e = 0
        self.esubopt_minus_Epf = 0
        self.sln_Epf = 0
        self.MFE = 0
        self.edesired_minus_MFE = 0
        self.recall = 0
        self.precision = 0
        self.edesired2 = 0
        self.edesired2_minus_Epf = 0

    # -- plain setters (the reference calls them get_*)
    def get_replica_num(self, rep_num):
        self.replica_num = rep_num

    def get_temp_shelf(self, temp):
        self.temp_shelf = temp

    def get_sim_step(self, step):
        self.sim_step = step

    def get_Epf(self, Epf):
        self.Epf = Epf

    def get_mfe_ss(self, ss):
        self.mfe_ss = ss

    def get_edesired(self, e_target):
        self.edesired = e_target

    def get_edesired_minus_Epf(self, Epf, e_target):
        self.edesired_minus_Epf = e_target - Epf

    def get_edesired2(self, e_target):
        self.edesired2 = e_target

    def get_edesired2_minus_Epf(self, Epf, e_target):
        self.edesired2_minus_Epf = e_target - Epf

    def get_subopt_e(self, e_subopt):
        self.subopt_e = e_subopt

    def get_esubopt_minus_Epf(self, Epf, e_subopt):
        self.esubopt_minus_Epf = e_subopt - Epf

    def get_precision(self, precision):
        self.precision = 1 - precision

    def get_recall(self, recall):
        self.recall = 1 - recall

    def get_mcc(self, mcc):
        self.mcc = 1 - mcc

    def get_mcc_alt(self, mcc_alt):
        self.mcc_alt = 1 - mcc_alt

    # -- derived terms
    def get_sln_Epf(self):
        self.sln_Epf = (self.Epf + 0.3759 * len(self.sequence) + 5.7534) / 10

    def get_MFE(self):
        self.MFE = RNA.fold(self.sequence)[1]

    def get_edesired_minus_MFE(self):
        self.edesired_minus_MFE = self.edesired - self.MFE

    def get_ensemble_defect(self, sec_struct):
        """energy_scores.py:362-374: fresh model details (bpp on), mfe, rescale, pf, ensemble_defect.  The engine
        runs MFE -> scaled inside -> outside -> defect in one call."""
        fc = RNA.fold_compound(self.sequence, RNA.md())
        (_, mfe) = fc.mfe()
        fc.exp_params_rescale(mfe)
        self.ensemble_defect = fc.ensemble_defect(sec_struct)

    def get_scoring_function(self, scoring_f):
        total = 0
        for function, weight in scoring_f:
            if function == "Ed-Epf":
                total += self.edesired_minus_Epf * weight
            elif function == "1-MCC":
                total += self.mcc * 10 * weight
            elif function == "sln_Epf":
                total += self.sln_Epf * weight
            elif function == "Ed-MFE":
                total += self.edesired_minus_MFE * weight
            elif function == "1-precision":
                total += self.precision * 10 * weight
            elif function == "1-recall":
                total += self.recall * 10 * weight
            elif function == "Edef":
                total += self.ensemble_defect * weight
        self.scoring_function = total

    def get_scoring_function_w_alt_ss(self):
        self.scoring_function = self.scoring_function + self.edesired2_minus_Epf

    def get_scoring_function_w_subopt(self):
        self.scoring_function = self.scoring_function - self.esubopt_minus_Epf

    def get_scoring_function_monomer(self, fc=None):
        """fc: the fold compound of sequence&sequence, if the caller folded it already (score_sequences)"""
        dimer = self.sequence + "&" + self.sequence
        if fc is None:
            fc = RNA.fold_compound(dimer)
        self.oligo_fraction = dme.oligo_fraction(dimer, fc)
        self.monomer_bonus = dme.kTlog_monomer_fraction(self.oligo_fraction)
        self.scoring_function = self.scoring_function + self.monomer_bonus

    def get_scoring_function_oligomer(self, fc):
        self.oligo_fraction = dme.oligo_fraction(self.sequence, fc)
        self.oligomer_bonus = dme.kTlog_oligo_fraction(self.oligo_fraction)
        self.scoring_function = self.scoring_function + self.oligomer_bonus

    def get_scoring_function_homomonomer(self, fc):
        self.oligo_fraction = dme.oligo_fraction(self.sequence, fc)
        self.oligomer_bonus = dme.kTlog_monomer_fraction(self.oligo_fraction)
        self.scoring_function = self.scoring_function + self.oligomer_bonus

    def update_scoring_function_w_motifs(self, motif_bonus):
        self.scoring_function += motif_bonus


def get_first_suboptimal_energy(sequence, a):
    """get_first_suboptimal_structure_and_energy(sequence, a, 1)[1] without the enumeration: the reference widens the band from 1 to
    49 kcal/mol until it holds two structures and takes the second of the sorted list -- i.e. the energy of the second-best
    structure if it lies within 49 kcal/mol of the MFE, else 0 (utils/energy_scores.py:476-488).  Single- and two-strand ('A&B')
    compounds alike; a compound without second_best_energy falls back to the enumeration."""
    if not hasattr(a, "second_best_energy"):
        return get_first_suboptimal_structure_and_energy(sequence, a, 1)[1]
    e1, e2 = a.second_best_energy()
    if e2 is None or round((e2 - e1) * 100.0) > 4900:
        return 0
    return e2


def get_first_suboptimal_structure_and_energy(sequence, a, number_of_suboptimals):
    """energy_scores.py:453-488: widen the energy band in 1 kcal/mol steps until the band holds enough structures,
    return the (k+1)-th best.  Needs fc.subopt_cb (Wuchty enumeration), which is outside the accelerated path
    (SURVEY.md 8f rank 3); the shim raises NotImplementedError."""
    RNA.cvar.uniq_ML = 1
    found = []

    def collect(structure, energy, data):
        if structure is not None:
            found.append([structure, energy])

    for band in range(100, 5000, 100):
        a.subopt_cb(band, collect, {"sequence": sequence})
        if len(found) >= number_of_suboptimals + 1:
            break
        found = []
    found.sort(key=lambda x: x[1])
    if not found:
        return "." * len(sequence), 0
    return found[number_of_suboptimals][0], found[number_of_suboptimals][1]
