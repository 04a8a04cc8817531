#include "ScoreSeqSet.h"

#include <algorithm>
#include <cassert>
#include <cmath>
#include <fstream>
#include <iomanip>
#include <iostream>

ScoreSeqSet::ScoreSeqSet( Motif* motif, BackgroundModel* bg, std::vector<Sequence*> seqSet )
    : motif_( motif ), bg_( bg ), seqSet_( seqSet ), Y_( motif->getY() ){}

ScoreSeqSet::~ScoreSeqSet(){}

// reference: ScoreSeqSet::calcLogOdds, src/seq_scoring/ScoreSeqSet.cpp:25-67
void ScoreSeqSet::calcLogOdds(){
    const size_t K = motif_->getK();
    const size_t W = motif_->getW();
    const size_t K_bg = ( bg_->getOrder() < K ) ? bg_->getOrder() : K;
    // the Motif's own table switches to log odds exactly as in the reference (callers read it through getS());
    // the device builds the identical table from v with the same libm logf
    motif_->calculateLogS( bg_->getV(), K_bg );

    const size_t N = seqSet_.size();
    zoops_scores_.assign( N, 0.0f );
    z_.assign( N, 0 );
    mops_off_.assign( N + 1, 0 );
    for( size_t n = 0; n < N; n++ ) mops_off_[n + 1] = mops_off_[n] + ( seqSet_[n]->getL() - W + 1 );
    if( keepMops_ ) mops_flat_.assign( mops_off_[N], 0.0f ); else mops_flat_.clear();
    if( N == 0 ) return;

    std::vector<uint64_t> indices;
    bool whole = false;
    SequenceSet* set = SequenceSet::commonSet( seqSet_, indices, &whole );
    std::vector<uint64_t> z64( N );
    BAMM_CHECK( bamm_score_logodds( set->device(), whole ? nullptr : indices.data(), N, static_cast<int>( W ), static_cast<int>( K ),
                                    static_cast<int>( bg_->getOrder() ), motif_->flatV().data(), bg_->flatV().data(),
                                    zoops_scores_.data(), z64.data(), keepMops_ ? mops_flat_.data() : nullptr ) );
    for( size_t n = 0; n < N; n++ ) z_[n] = static_cast<size_t>( z64[n] );
}

std::vector<std::vector<float>> ScoreSeqSet::getMopsScores(){
    std::vector<std::vector<float>> out( seqSet_.size() );
    if( mops_flat_.empty() ) return out;
    for( size_t n = 0; n < seqSet_.size(); n++ ){
        out[n].assign( mops_flat_.begin() + mops_off_[n], mops_flat_.begin() + mops_off_[n + 1] );
    }
    return out;
}

// Rank p-values of window scores against the sorted negative scores with an exponential tail for the top ranks
// (reference: ScoreSeqSet::calcPvalues, src/seq_scoring/ScoreSeqSet.cpp:70-126)
void ScoreSeqSet::calcPvalues( std::vector<std::vector<float>> pos_scores, std::vector<float> neg_all_scores ){
    // The sort of all negative window scores and the per-window rank search run on the device (bamm_mops_pvalues restates
    // ScoreSeqSet.cpp:85-124: ascending sort, rate parameter from the first nTop sorted values, upper_bound per window,
    // exponential tail / linear interpolation); the host only flattens and scatters the vectors.
    const size_t posN = seqSet_.size();
    mops_p_values_.assign( posN, std::vector<float>() );
    mops_e_values_.assign( posN, std::vector<float>() );
    std::vector<uint64_t> off( posN + 1, 0 );
    for( size_t n = 0; n < posN; n++ ){
        const size_t LW1 = seqSet_[n]->getL() - motif_->getW() + 1;
        if( pos_scores[n].size() < LW1 ){
            std::cerr << "Error: calcPvalues needs the scores of every window (sequence " << n << ")." << std::endl;
            exit( 1 );
        }
        off[n + 1] = off[n] + LW1;
    }
    std::vector<float> flat( off[posN] ), p( off[posN] ), e( off[posN] );
    for( size_t n = 0; n < posN; n++ ) std::copy( pos_scores[n].begin(), pos_scores[n].begin() + ( off[n + 1] - off[n] ), flat.begin() + off[n] );
    BAMM_CHECK( bamm_mops_pvalues( neg_all_scores.data(), neg_all_scores.size(), flat.data(), flat.size(), posN, p.data(), e.data() ) );
    for( size_t n = 0; n < posN; n++ ){
        mops_p_values_[n].assign( p.begin() + off[n], p.begin() + off[n + 1] );
        mops_e_values_[n].assign( e.begin() + off[n], e.begin() + off[n + 1] );
    }
    pval_is_calulated_ = true;
}

void ScoreSeqSet::printLogOdds(){
    for( size_t n = 0; n < seqSet_.size(); n++ ){
        std::cout << "seq " << n << ":" << std::endl << zoops_scores_[n] << '\t';
        for( size_t i = mops_off_[n]; i < mops_off_[n + 1] && i < mops_flat_.size(); i++ ) std::cout << mops_flat_[i] << '\t';
        std::cout << std::endl;
    }
}

// BaMMScan: the negative window scores are computed and sorted on the device once for this motif, the positive windows are
// scored and given their p-values there, and only the windows with p < pvalCutoff come back (in sequence order, window
// ascending) - the same windows and values as calcLogOdds + calcPvalues + the filter of write()
void ScoreSeqSet::scanOccurrences( const std::vector<Sequence*>& negSet, float pvalCutoff ){
    const int W = static_cast<int>( motif_->getW() ), K = static_cast<int>( motif_->getK() );
    std::vector<uint64_t> negIdx, posIdx;
    bool negWhole = false, posWhole = false;
    SequenceSet* neg = SequenceSet::commonSet( negSet, negIdx, &negWhole );
    SequenceSet* pos = SequenceSet::commonSet( seqSet_, posIdx, &posWhole );
    bamm_scan* scan = nullptr;
    BAMM_CHECK( bamm_scan_create( neg->device(), negWhole ? nullptr : negIdx.data(), negSet.size(), W, K, static_cast<int>( bg_->getOrder() ),
                                  motif_->flatV().data(), bg_->flatV().data(), &scan ) );
    hits_.clear();
    const uint64_t page = 1u << 20;
    uint64_t cursor = 0, got = page;
    while( got == page ){
        const size_t have = hits_.size();
        hits_.resize( have + page );
        BAMM_CHECK( bamm_scan_hits( scan, pos->device(), posWhole ? nullptr : posIdx.data(), seqSet_.size(), seqSet_.size(), pvalCutoff,
                                    &cursor, hits_.data() + have, page, &got ) );
        hits_.resize( have + got );
    }
    bamm_scan_destroy( scan );
    hits_are_scanned_ = true;
}

// one line of the .occurrence file: window i of sequence n (reference: ScoreSeqSet.cpp:245-291)
void ScoreSeqSet::writeOccurrence( std::ostream& ofile, size_t n, size_t i, float p, float e, bool ss ){
    size_t seqlen = seqSet_[n]->getL();
    if( !ss ) seqlen = ( seqlen - 1 ) / 2;
    const size_t end = i + motif_->getW();
    const uint8_t* codes = seqSet_[n]->getSequence();
    ofile << seqSet_[n]->getHeader() << '\t' << seqlen << '\t' << ( ( i < seqlen ) ? '+' : '-' ) << '\t'
          << i + 1 << ".." << end << '\t';
    for( size_t m = i; m < end; m++ ) ofile << Alphabet::getBase( codes[m] );
    ofile << '\t' << std::setprecision( 3 ) << p << '\t' << e << '\n';
}

// .occurrence (reference: ScoreSeqSet::write, src/seq_scoring/ScoreSeqSet.cpp:245-291): from the p-values of calcPvalues, or
// from the hits of scanOccurrences
void ScoreSeqSet::write( char* odir, std::string basename, float pvalCutoff, bool ss ){
    assert( pval_is_calulated_ || hits_are_scanned_ );
    std::ofstream ofile( std::string( odir ) + '/' + basename + ".occurrence" );
    ofile << "seq\tlength\tstrand\tstart..end\tpattern\tp-value\te-value" << std::endl;
    if( !pval_is_calulated_ ){
        for( const bamm_hit& h : hits_ )
            if( h.p_value < pvalCutoff ) writeOccurrence( ofile, h.seq, h.window, h.p_value, h.e_value, ss );
        return;
    }
    const size_t W = motif_->getW();
    for( size_t n = 0; n < seqSet_.size(); n++ ){
        const size_t LW1 = seqSet_[n]->getL() - W + 1;
        for( size_t i = 0; i < LW1; i++ )
            if( mops_p_values_[n][i] < pvalCutoff ) writeOccurrence( ofile, n, i, mops_p_values_[n][i], mops_e_values_[n][i], ss );
    }
}

// .logOddsZoops (reference: ScoreSeqSet::writeLogOdds, src/seq_scoring/ScoreSeqSet.cpp:293-331)
void ScoreSeqSet::writeLogOdds( char* odir, std::string basename, bool ss ){
    std::ofstream ofile( std::string( odir ) + '/' + basename + ".logOddsZoops" );
    ofile << "seq\tlength\tstrand\tstart..end\tpattern\tzoops_score" << std::endl;
    const size_t W = motif_->getW();
    for( size_t n = 0; n < seqSet_.size(); n++ ){
        size_t seqlen = seqSet_[n]->getL();
        if( !ss ) seqlen = ( seqlen - 1 ) / 2;
        const uint8_t* codes = seqSet_[n]->getSequence();
        const size_t end = z_[n] + W;
        ofile << seqSet_[n]->getHeader() << '\t' << seqlen << '\t' << ( ( z_[n] < seqlen ) ? '+' : '-' ) << '\t'
              << z_[n] + 1 << ".." << end << '\t';
        for( size_t m = z_[n]; m < end; m++ ) ofile << Alphabet::getBase( codes[m] );
        ofile << '\t' << std::setprecision( 3 ) << zoops_scores_[n] << '\n';
    }
}
