// BaMMScan driver on the B200 path: scans a sequence set with every motif of a model file and writes the windows whose
// p-value against a sampled background set is below --pvalCutoff (<basename>_motif_<n>.occurrence). The flow is that of
// mainBaMM.cpp without EM: background model, initial motifs, sequences shorter than the widest motif dropped, the negative
// set sampled once and shared by all motifs, then per motif the device scan (ScoreSeqSet::scanOccurrences). The files are
// those `BaMMmotif ... --scoreSeqset` writes for the same model, background and sequences. Options: Global (scan mode).
#include <chrono>
#include <cstdlib>
#include <iostream>
#include <memory>
#include <vector>

#include "Global.h"
#include "MotifSet.h"
#include "ScoreSeqSet.h"
#include "SeqGenerator.h"
#include "Util.h"

int main( int nargs, char* args[] ){
    auto t0_wall = std::chrono::high_resolution_clock::now();
    std::cout << std::endl
              << "======================================" << std::endl
              << "=      Welcome to use BaMMScan       =" << std::endl
              << "=          Version 2.0 (B200 path)   =" << std::endl
              << "======================================" << std::endl;

    util::srand42( 42 );                                    // the N draws of the FASTA reader follow, as in mainBaMM.cpp
    const char* dev = getenv( "BAMM_DEVICE" );
    if( dev && atoi( dev ) != 0 ) BAMM_CHECK( bamm_set_device( atoi( dev ) ) );
    Global::init( nargs, args, true );
    if( Global::initialModelTag == "BaMM" && !Global::bgModelGiven ){
        std::cout << "No background Model file provided for initial search motif!\n";
        exit( 1 );
    }

    std::vector<Sequence*> posSet = Global::posSequenceSet->getSequences();
    BackgroundModel* bgModel = Global::bgModelGiven
        ? new BackgroundModel( Global::bgModelFilename )
        : new BackgroundModel( posSet, Global::bgModelOrder, Global::bgModelAlpha, Global::interpolateBG, Global::outputFileBasename );

    MotifSet motif_set( Global::initialModelFilename, Global::addColumns.at( 0 ), Global::addColumns.at( 1 ), Global::initialModelTag,
                        Global::posSequenceSet, bgModel->getV(), Global::bgModelOrder, Global::modelOrder, Global::modelAlpha,
                        Global::maxPWM, Global::q );

    {
        std::vector<Sequence*> kept;
        for( Sequence* s : posSet ) if( s->getL() >= motif_set.getMaxW() ) kept.push_back( s );
        posSet.swap( kept );
    }
    if( posSet.empty() ){
        std::cerr << "There are 0 sequences longer than input motif. Exit!\n";
        exit( 1 );
    }
    const size_t minSeqN = 5000;                            // the mFold rule of mainBaMM.cpp
    const bool rest = minSeqN % posSet.size();
    if( posSet.size() < minSeqN ) Global::mFold = minSeqN / posSet.size() + rest;

    SeqGenerator negseq( posSet, NULL, Global::sOrder, 1.0f, Global::genericNeg );
    std::unique_ptr<SequenceSet> negSequences = negseq.sample_bgseqset_by_fold( Global::mFold );
    std::vector<Sequence*> negSet = negSequences->getSequences();

    for( size_t n = 0; n < motif_set.getN(); n++ ){
        Motif* motif = new Motif( *motif_set.getMotifs()[n] );
        const std::string motifName = Global::outputFileBasename + "_motif_" + std::to_string( n + 1 );
        if( Global::saveLogOdds ){                          // the ZOOPS files of --scoreSeqset --saveLogOdds
            ScoreSeqSet scoreNegSet( motif, bgModel, negSet );
            scoreNegSet.setKeepMops( false );
            scoreNegSet.calcLogOdds();
            scoreNegSet.writeLogOdds( Global::outputDirectory, Global::outputFileBasename + ".negSet", Global::ss );
            ScoreSeqSet scorePosSet( motif, bgModel, posSet );
            scorePosSet.setKeepMops( false );
            scorePosSet.calcLogOdds();
            scorePosSet.writeLogOdds( Global::outputDirectory, motifName, Global::ss );
        }
        ScoreSeqSet scan( motif, bgModel, posSet );
        scan.scanOccurrences( negSet, Global::pvalCutoff );
        scan.write( Global::outputDirectory, motifName, Global::pvalCutoff, Global::ss );
        std::cout << "motif " << n + 1 << ": " << scan.getHits().size() << " occurrences with p < " << Global::pvalCutoff << std::endl;
        delete motif;
    }

    auto t_diff = std::chrono::duration_cast<std::chrono::duration<double>>( std::chrono::high_resolution_clock::now() - t0_wall );
    std::cout << std::endl << "------ Runtime: " << t_diff.count() << " seconds -------" << std::endl;
    negSequences.reset();
    delete bgModel;
    Global::destruct();
    return 0;
}
