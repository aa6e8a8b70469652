/*
 * cPecanEm -- trains the pair-HMM by expectation maximisation over a set of pairwise alignments (cigars on stdin) of the
 * sequences in the FASTA files given, and writes the model file that cPecanRealign --loadHmm reads.
 *
 * It is the reference's cPecanEm.py (expectationMaximisation / calculateMaximisation / expectationMaximisationTrials,
 * cPecanEm.py:112-242) without jobTree: there every iteration starts one cPecanRealign --outputExpectations subprocess per
 * alignment file, sums the expectation files and normalises in Python; here the alignments go to the device once
 * (cpecanResidentBatch) and an iteration is one expectation pass of the engine (cell_calculateExpectation's path,
 * impl/pairwiseAligner.c:418-438, :735-746) followed by the same maximisation step on the host:
 *     normalise -> [keep the old emissions unless --trainEmissions; --tieEmissions] -> next model.
 * Same options where they make sense in one process; the model file is written in cPecanEm.py's format (:31-35): line 1 type,
 * transitions, likelihood; line 2 emissions; line 3 the likelihood of every iteration.
 * --updateTheBand: after the maximisation step of every iteration but the last, every alignment is realigned under the model that step
 * produced and re-anchored from the result, so that the next expectation pass runs in a band that follows the model rather than the
 * input cigars.  The order is train, then re-anchor under the new model; the band is never derived from the untrained starting model
 * (under all-equal or random values a realignment says nothing).  One update is what cPecanRealign --loadHmm <model>
 * --diagonalExpansion 10 --splitMatrixBiggerThanThis 3000 --constraintDiagonalTrim t (matchGamma 0.85, its default) writes for the
 * current alignments, read back by cPecanEm -- but under the model in full doubles rather than through the model file's 12 digits, and on
 * the device (cpecanResidentBatch_updateAnchors): no list, alignment or cigar crosses to the host.  Every --randomStart trial starts from
 * the input alignments' anchors.
 * Not carried over: the XML summary and the LASTZ scoring-matrix export.
 * Several GPUs: tools/em_multi_gpu.py runs the same loop with one NCCL all-reduce of the expectation vector per iteration.
 */
#include <getopt.h>
#include <math.h>
#include <time.h>

#include "realignJobs.h"

static void usage(void) {
    fprintf(stderr, "cPecanEm [options] seq1[fasta] [seq2[fasta] ...] < alignments.cigar\n");
    fprintf(stderr, "Trains the pair-HMM on the given alignments by expectation maximisation (B200 batched engine)\n");
    fprintf(stderr, "--logLevel L : INFO / DEBUG\n");
    fprintf(stderr, "--inputModel FILE : start from this model\n");
    fprintf(stderr, "--outputModel FILE : where the trained model goes (default hmm.txt)\n");
    fprintf(stderr, "--modelType T : fiveState (default), fiveStateAsymmetric, threeState, threeStateAsymmetric\n");
    fprintf(stderr, "--iterations N : iterations of EM (default 10)\n");
    fprintf(stderr, "--randomStart : start from small random values, else from all-equal values\n");
    fprintf(stderr, "--trials N : independent trials with --randomStart; the model with the highest likelihood is kept (default 3)\n");
    fprintf(stderr, "--outputTrialHmms : also write every trial's model, as outputModel_i\n");
    fprintf(stderr, "--useDefaultModelAsStart : the first iteration's expectations come from the built-in model\n");
    fprintf(stderr, "--setJukesCantorStartingEmissions D : starting emissions from the Jukes-Cantor expectation at D substitutions per site\n");
    fprintf(stderr, "--trainEmissions : train the emissions as well as the transitions\n");
    fprintf(stderr, "--tieEmissions : with --trainEmissions, emissions only distinguish match from mismatch\n");
    fprintf(stderr, "--maxAlignmentLengthToSample N : use at most N bases of alignment, sampled without replacement (default 50000000)\n");
    fprintf(stderr, "--seed N : seed of the random start and of the sampling (default: time)\n");
    fprintf(stderr, "--gpus N : spread the alignments over the first N GPUs; the expectations are summed with one NCCL all-reduce per iteration (default 1)\n");
    fprintf(stderr, "--updateTheBand : after every iteration but the last, realign the alignments under the new model (as cPecanRealign, matchGamma 0.85)\n");
    fprintf(stderr, "    and take the next iteration's anchors from the realigned alignments\n");
    fprintf(stderr, "--diagonalExpansion N, --constraintDiagonalTrim N, --splitMatrixBiggerThanThis N : band options, as cPecanRealign\n");
    fprintf(stderr, "    (defaults: cPecanEm.py's --optionsToRealign, diagonalExpansion 10 and splitMatrixBiggerThanThis 3000)\n");
}

static StateMachineType model_type(const char *name) {
    if (strcmp(name, "fiveState") == 0) return fiveState;
    if (strcmp(name, "fiveStateAsymmetric") == 0) return fiveStateAsymmetric;
    if (strcmp(name, "threeState") == 0) return threeState;
    if (strcmp(name, "threeStateAsymmetric") == 0) return threeStateAsymmetric;
    st_errAbort("cPecanEm: unknown model type %s", name);
    return fiveState;
}

/* cPecanEm.py:31-35, numbers with 12 significant digits as Python 2's str() prints them; then the running likelihoods (:170-173) */
static void write_model(const Hmm *hmm, const char *file, const double *likelihoods, int64_t nLikelihoods) {
    FILE *f = fopen(file, "w");
    if (f == NULL) st_errAbort("cPecanEm: cannot write %s", file);
    const int64_t S = hmm->stateNumber;
    fprintf(f, "%d", (int) hmm->type);
    for (int64_t i = 0; i < S * S; i++) fprintf(f, " %.12g", hmm->transitions[i]);
    fprintf(f, " %.12g\n", hmm->likelihood);
    for (int64_t i = 0; i < S * 16; i++) fprintf(f, "%s%.12g", i ? " " : "", hmm->emissions[i]);
    fprintf(f, "\n");
    if (likelihoods != NULL) {
        for (int64_t i = 0; i < nLikelihoods; i++) fprintf(f, "%s%.12g", i ? "\t" : "", likelihoods[i]);
        fprintf(f, "\n");
    }
    fclose(f);
}

static void equalise(Hmm *hmm) { /* cPecanEm.py:81-85 */
    const int64_t S = hmm->stateNumber;
    for (int64_t i = 0; i < S * S; i++) hmm->transitions[i] = 1.0 / (double) S;
    for (int64_t i = 0; i < S * 16; i++) hmm->emissions[i] = 1.0 / 16.0;
}

static void jukes_cantor_emissions(Hmm *hmm, double divergence) { /* cPecanEm.py:87-93; the only exponential on the host side */
    const double e = exp(-4.0 * divergence / 3.0), same = (0.25 + 0.75 * e) / 4.0, different = (0.25 - 0.25 * e) / 4.0;
    for (int64_t s = 0; s < hmm->stateNumber; s++) {
        for (int x = 0; x < 4; x++) {
            for (int y = 0; y < 4; y++) hmm->emissions[s * 16 + x * 4 + y] = x == y ? same : different;
        }
    }
}

static void tie_emissions(Hmm *hmm) { /* cPecanEm.py:95-105 */
    for (int64_t s = 0; s < hmm->stateNumber; s++) {
        double *e = hmm->emissions + s * 16, identity = 0.0;
        for (int x = 0; x < 4; x++) identity += e[x * 4 + x];
        for (int x = 0; x < 4; x++) {
            for (int y = 0; y < 4; y++) e[x * 4 + y] = x == y ? identity / 4.0 : (1.0 - identity) / 12.0;
        }
    }
}

/* the matchGamma of cPecanRealign's default realignment (cPecanRealign.c, o.matchGamma) with which --updateTheBand realigns */
#define UPDATE_BAND_MATCH_GAMMA 0.85f

typedef struct {
    const char *inputModel;
    StateMachineType type;
    int64_t iterations;
    bool randomStart, useDefaultModelAsStart, trainEmissions, tieEmissions, updateTheBand;
    double jukesCantor; /* < 0: not set */
} EmOptions;

/* one EM run (cPecanEm.py:112-215); returns the trained model, hmm->likelihood = that of the last iteration */
static Hmm *expectation_maximisation(CpecanResidentBatch *batch, PairwiseAlignmentParameters *p, const EmOptions *o, const char *outputModel,
                                     double *likelihoods) {
    Hmm *hmm;
    if (o->inputModel != NULL) {
        log_info("Loading the model from the input file %s\n", o->inputModel);
        hmm = hmm_loadFromFile(o->inputModel);
        hmm_normalise(hmm);
    } else {
        hmm = hmm_constructEmpty(0.0, o->type);
        if (o->randomStart) hmm_randomise(hmm);
        else equalise(hmm);
    }
    if (o->jukesCantor >= 0.0) jukes_cantor_emissions(hmm, o->jukesCantor);
    write_model(hmm, outputModel, NULL, 0);
    for (int64_t it = 0; it < o->iterations; it++) {
        StateMachine *sM;
        if (o->useDefaultModelAsStart && it == 0) {
            sM = hmm->stateNumber == 5 ? stateMachine5_construct(hmm->type) : stateMachine3_construct(hmm->type);
        } else {
            sM = hmm_getStateMachine(hmm);
        }
        Hmm *expectations = hmm_constructEmpty(0.000000000001, hmm->type); /* the tiny pseudo-count prevents overflow (cPecanRealign.c:493) */
        cpecanResidentBatch_getExpectations(batch, sM, expectations, p);
        stateMachine_destruct(sM);
        hmm_normalise(expectations);
        likelihoods[it] = expectations->likelihood;
        log_info("On %" PRIi64 " iteration got likelihood: %.12g\n", it, expectations->likelihood);
        if (o->trainEmissions) {
            if (o->tieEmissions) tie_emissions(expectations);
        } else {
            memcpy(expectations->emissions, hmm->emissions, (size_t) hmm->stateNumber * 16 * sizeof(double));
        }
        hmm_destruct(hmm);
        hmm = expectations;
        write_model(hmm, outputModel, NULL, 0);
        if (o->updateTheBand && it + 1 < o->iterations) { /* the next iteration's band, from the alignments under the model just trained */
            sM = hmm_getStateMachine(hmm);
            cpecanResidentBatch_updateAnchors(batch, sM, p, UPDATE_BAND_MATCH_GAMMA);
            stateMachine_destruct(sM);
            log_info("Updated the band under the model of iteration %" PRIi64 "\n", it);
        }
    }
    write_model(hmm, outputModel, likelihoods, o->iterations);
    return hmm;
}

static void release_jobs(Job *jobs, int64_t n, const char **sX, const char **sY, stList **anchors, bool *ragged) {
    for (int64_t i = 0; i < n; i++) job_release(&jobs[i]);
    free(jobs);
    free(sX);
    free(sY);
    free(anchors);
    free(ragged);
}

int main(int argc, char *argv[]) {
    PairwiseAlignmentParameters *p = pairwiseAlignmentBandingParameters_construct();
    p->constraintDiagonalTrim = 0; /* cPecanRealign's defaults, then cPecanEm.py:371 */
    p->diagonalExpansion = 10;
    p->splitMatrixBiggerThanThis = (int64_t) 3000 * 3000;
    EmOptions o;
    memset(&o, 0, sizeof(o));
    o.type = fiveState;
    o.iterations = 10;
    o.jukesCantor = -1.0;
    const char *outputModel = "hmm.txt";
    int64_t trials = 3, maxSample = 50000000;
    bool outputTrialHmms = false;
    long seed = (long) time(NULL);

    static struct option longOptions[] = { { "logLevel", required_argument, 0, 'a' },
                                           { "help", no_argument, 0, 'h' },
                                           { "inputModel", required_argument, 0, 'I' },
                                           { "outputModel", required_argument, 0, 'O' },
                                           { "modelType", required_argument, 0, 'M' },
                                           { "iterations", required_argument, 0, 'n' },
                                           { "trials", required_argument, 0, 'T' },
                                           { "outputTrialHmms", no_argument, 0, 'H' },
                                           { "randomStart", no_argument, 0, 'R' },
                                           { "useDefaultModelAsStart", no_argument, 0, 'D' },
                                           { "setJukesCantorStartingEmissions", required_argument, 0, 'J' },
                                           { "trainEmissions", no_argument, 0, 'E' },
                                           { "tieEmissions", no_argument, 0, 'e' },
                                           { "maxAlignmentLengthToSample", required_argument, 0, 'S' },
                                           { "seed", required_argument, 0, 's' },
                                           { "diagonalExpansion", required_argument, 0, 'r' },
                                           { "constraintDiagonalTrim", required_argument, 0, 't' },
                                           { "splitMatrixBiggerThanThis", required_argument, 0, 'o' },
                                           { "gpus", required_argument, 0, 'G' },
                                           { "updateTheBand", no_argument, 0, 'U' },
                                           { 0, 0, 0, 0 } };
    for (;;) {
        int index = 0;
        const int key = getopt_long(argc, argv, "a:hr:t:o:", longOptions, &index);
        if (key == -1) break;
        switch (key) {
        case 'a': set_log_level(optarg); break;
        case 'h': usage(); return 0;
        case 'I': o.inputModel = optarg; break;
        case 'O': outputModel = optarg; break;
        case 'M': o.type = model_type(optarg); break;
        case 'n': o.iterations = parse_int(optarg, "--iterations"); break;
        case 'T': trials = parse_int(optarg, "--trials"); break;
        case 'H': outputTrialHmms = true; break;
        case 'R': o.randomStart = true; break;
        case 'D': o.useDefaultModelAsStart = true; break;
        case 'J': o.jukesCantor = parse_float(optarg, "--setJukesCantorStartingEmissions"); break;
        case 'E': o.trainEmissions = true; break;
        case 'e': o.tieEmissions = true; break;
        case 'S': maxSample = parse_int(optarg, "--maxAlignmentLengthToSample"); break;
        case 's': seed = (long) parse_int(optarg, "--seed"); break;
        case 'r':
            p->diagonalExpansion = parse_int(optarg, "--diagonalExpansion");
            if (p->diagonalExpansion % 2 != 0) st_errAbort("cPecanEm: --diagonalExpansion must be even");
            break;
        case 't': p->constraintDiagonalTrim = parse_int(optarg, "--constraintDiagonalTrim"); break;
        case 'o': {
            const int64_t side = parse_int(optarg, "--splitMatrixBiggerThanThis");
            p->splitMatrixBiggerThanThis = side * side;
            break;
        }
        case 'G': {
            const int64_t gpus = parse_int(optarg, "--gpus");
            if (gpus < 1 || gpus > 16) st_errAbort("cPecanEm: --gpus takes 1 to 16");
            cpecan_setDevices((int) gpus);
            break;
        }
        case 'U': o.updateTheBand = true; break;
        default: usage(); return 1;
        }
    }
    if (optind >= argc) {
        usage();
        return 1;
    }
    srand48(seed);
    read_sequence_files(argc, argv, optind);

    /* All alignments are read, shuffled (so that a sample is not just the head of the file) and sampled up to maxSample bases of
     * alignment length (cPecanEm.py:148-160); only the sampled ones have their sub-sequences cut and their anchors built. */
    struct PairwiseAlignment **all = NULL;
    int64_t n = 0, cap = 0;
    struct PairwiseAlignment *pA;
    while ((pA = cigarRead(stdin)) != NULL) {
        if (n == cap) {
            cap = cap ? 2 * cap : 1024;
            all = realloc(all, (size_t) cap * sizeof(*all));
            if (all == NULL) st_errAbort("cPecanEm: out of memory");
        }
        all[n++] = pA;
    }
    if (n == 0) st_errAbort("cPecanEm: no alignments on the standard input");
    for (int64_t i = n - 1; i > 0; i--) {
        const int64_t k = (int64_t) (drand48() * (double) (i + 1));
        struct PairwiseAlignment *t = all[i];
        all[i] = all[k];
        all[k] = t;
    }
    int64_t used = 0;
    double sampled = 0.0;
    while (used < n && sampled < (double) maxSample) {
        sampled += (double) (llabs((long long) (all[used]->end1 - all[used]->start1)) + llabs((long long) (all[used]->end2 - all[used]->start2))) / 2.0;
        used++;
    }
    log_info("We sampled: %.0f bases of alignment length and %" PRIi64 " alignments of %" PRIi64 "\n", sampled, used, n);
    Job *jobs = xmalloc((size_t) used * sizeof(Job));
    for (int64_t i = 0; i < used; i++) job_prepare(&jobs[i], all[i], p);
    for (int64_t i = used; i < n; i++) destructPairwiseAlignment(all[i]);
    free(all);
    const char **sX = xmalloc((size_t) used * sizeof(char *)), **sY = xmalloc((size_t) used * sizeof(char *));
    stList **anchors = xmalloc((size_t) used * sizeof(stList *));
    bool *ragged = xmalloc((size_t) used * sizeof(bool));
    for (int64_t i = 0; i < used; i++) {
        sX[i] = jobs[i].subX;
        sY[i] = jobs[i].subY;
        anchors[i] = jobs[i].filtered;
        ragged[i] = 1;
    }
    CpecanResidentBatch *batch = cpecanResidentBatch_construct(used, sX, sY, anchors, p, ragged, ragged);
    free_sequences(); /* the jobs hold their own sub-sequences */
    if (!o.updateTheBand) release_jobs(jobs, used, sX, sY, anchors, ragged); /* else kept: every trial starts from the input alignments' anchors */

    double *likelihoods = xmalloc((size_t) (o.iterations + 1) * sizeof(double));
    if (o.inputModel != NULL || !o.randomStart) { /* one run (cPecanEm.py:218-219) */
        Hmm *hmm = expectation_maximisation(batch, p, &o, outputModel, likelihoods);
        log_info("Trained model has likelihood %.12g\n", hmm->likelihood);
        hmm_destruct(hmm);
    } else {
        log_info("Running %" PRIi64 " random restart trials to find best hmm\n", trials);
        Hmm *best = NULL;
        double *bestLikelihoods = xmalloc((size_t) (o.iterations + 1) * sizeof(double));
        char *trialFile = xmalloc(strlen(outputModel) + 32);
        for (int64_t t = 0; t < trials; t++) {
            sprintf(trialFile, "%s_%" PRIi64, outputModel, t);
            if (o.updateTheBand && t > 0) { /* the previous trial moved the band */
                cpecanResidentBatch_destruct(batch);
                batch = cpecanResidentBatch_construct(used, sX, sY, anchors, p, ragged, ragged);
            }
            Hmm *hmm = expectation_maximisation(batch, p, &o, trialFile, likelihoods);
            if (!outputTrialHmms) remove(trialFile);
            if (best == NULL || hmm->likelihood > best->likelihood) {
                if (best != NULL) hmm_destruct(best);
                best = hmm;
                memcpy(bestLikelihoods, likelihoods, (size_t) o.iterations * sizeof(double));
            } else {
                hmm_destruct(hmm);
            }
        }
        if (best != NULL) {
            log_info("Hmm with highest likelihood: %.12g\n", best->likelihood);
            write_model(best, outputModel, bestLikelihoods, o.iterations);
            hmm_destruct(best);
        }
        free(bestLikelihoods);
        free(trialFile);
    }
    free(likelihoods);
    cpecanResidentBatch_destruct(batch);
    if (o.updateTheBand) release_jobs(jobs, used, sX, sY, anchors, ragged);
    pairwiseAlignmentBandingParameters_destruct(p);
    cpecan_shutdown();
    return 0;
}
