// ScoreSeqSet — log-odds scoring of every window of a sequence list; host wrapper over bamm_score_logodds().
// Public interface = the reference's (src/seq_scoring/ScoreSeqSet.h:24-37). MOPS scores (one per window) are kept
// flat; setKeepMops(false) skips materialising them when only ZOOPS scores are consumed (FDR's default).
// scanOccurrences() is the route of BaMMScan: the negative scores stay on the device and only the hits come back.
#ifndef BAMM_HOST_SCORESEQSET_H_
#define BAMM_HOST_SCORESEQSET_H_

#include <string>
#include <vector>

#include "BackgroundModel.h"
#include "Motif.h"

class ScoreSeqSet {
public:
    ScoreSeqSet( Motif* motif, BackgroundModel* bg, std::vector<Sequence*> seqSet );
    ~ScoreSeqSet();

    void setKeepMops( bool keep )   { keepMops_ = keep; }
    void calcLogOdds();
    void calcPvalues( std::vector<std::vector<float>> pos_mops_scores, std::vector<float> neg_all_scores );
    // the windows with p < pvalCutoff, p against every window of negSet, all on the device (bamm_scan_*); write() then
    // writes these hits
    void scanOccurrences( const std::vector<Sequence*>& negSet, float pvalCutoff );
    const std::vector<bamm_hit>&    getHits() const     { return hits_; }

    std::vector<std::vector<float>> getMopsScores();
    std::vector<float>              getZoopsScores()    { return zoops_scores_; }
    const std::vector<float>&       flatMopsScores() const { return mops_flat_; }
    const std::vector<size_t>&      getZ() const        { return z_; }

    void write( char* odir, std::string basename, float pvalCutoff, bool ss );
    void writeLogOdds( char* odir, std::string basename, bool ss );
    void printLogOdds();

private:
    void writeOccurrence( std::ostream& out, size_t n, size_t i, float p, float e, bool ss );

    Motif*                          motif_;
    BackgroundModel*                bg_;
    std::vector<Sequence*>          seqSet_;
    bool                            keepMops_ = true;

    std::vector<float>              zoops_scores_;
    std::vector<float>              mops_flat_;         // all window scores, sequence after sequence
    std::vector<size_t>             mops_off_;          // nseq+1 offsets into mops_flat_
    std::vector<std::vector<float>> mops_p_values_;
    std::vector<std::vector<float>> mops_e_values_;
    std::vector<size_t>             z_;
    bool                            pval_is_calulated_ = false;
    std::vector<bamm_hit>           hits_;
    bool                            hits_are_scanned_ = false;
    std::vector<size_t>             Y_;
};

#endif
