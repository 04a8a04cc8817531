// Global — command-line options of the BaMMmotif driver (static singleton like the reference's,
// src/refinement/Global.h). Flag names, defaults and the presence-overwrites-default behaviour of boolean flags follow
// src/refinement/Global.cpp:6-96, 120-344 — NOT the README (SURVEY.md A9, A15).
#ifndef BAMM_HOST_GLOBAL_H_
#define BAMM_HOST_GLOBAL_H_

#include <limits>
#include <string>
#include <vector>

#include "SequenceSet.h"

class Global {
public:
    // scan: the options of BaMMScan (mainScan.cpp): -m/--mFold and -s/--sOrder without --FDR, no training or evaluation
    // options, and a single input sequence is enough
    static void init( int nargs, char* args[], bool scan = false );
    static void destruct();
    static void printHelp();
    static void printStat();

    static char*        outputDirectory;
    static std::string  outputFileBasename;
    static char*        posSequenceFilename;
    static std::string  posSequenceBasename;
    static SequenceSet* posSequenceSet;
    static char*        negSequenceFilename;
    static std::string  negSequenceBasename;
    static SequenceSet* negSequenceSet;
    static bool         negSeqGiven;
    static bool         genericNeg;
    static std::string  alphabetType;
    static bool         ss;

    static char*        initialModelFilename;
    static std::string  initialModelBasename;
    static std::string  initialModelTag;
    static size_t       maxPWM;
    static bool         mops;
    static bool         zoops;

    static size_t               modelOrder;
    static std::vector<float>   modelAlpha;
    static float                modelBeta;
    static float                modelGamma;
    static std::vector<size_t>  addColumns;
    static bool                 interpolateBG;

    static char*                bgModelFilename;
    static bool                 bgModelGiven;
    static size_t               bgModelOrder;
    static std::vector<float>   bgModelAlpha;

    static bool         EM;
    static float        q;
    static bool         optimizeQ;
    static float        f;
    static bool         CGS;
    static bool         advanceEM;

    static bool         FDR;
    static size_t       mFold;
    static size_t       cvFold;
    static size_t       sOrder;

    static bool         scoreSeqset;
    static float        pvalCutoff;

    static bool         verbose;
    static bool         debugMode;
    static bool         saveBaMMs;
    static bool         savePRs;
    static bool         savePvalues;
    static bool         saveLogOdds;
    static bool         saveInitialBaMMs;
    static bool         saveBgModel;

    static size_t       threads;

private:
    static int  readArguments( int nargs, char* args[], bool scan );
};

#endif
