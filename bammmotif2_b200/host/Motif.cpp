#include "Motif.h"
#include "Device.h"

#include <cmath>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <limits>
#include <random>
#include <sstream>

#include "Util.h"

void Motif::allocate(){
    Y_.clear();
    for( size_t k = 0; k < K_ + 8; k++ ) Y_.push_back( util::ipow( Alphabet::getSize(), k ) );
    off_.assign( K_ + 2, 0 );
    for( size_t k = 0; k <= K_; k++ ) off_[k + 1] = off_[k] + Y_[k + 1] * W_;
    v_.assign( off_[K_ + 1], 0.0f );
    p_.assign( off_[K_ + 1], 0.0f );
    n_.assign( off_[K_ + 1], 0 );
    a_.assign( ( K_ + 1 ) * W_, 0.0f );
    s_.assign( Y_[K_ + 1] * W_, 0.0f );
}

void Motif::bindViews(){
    size_t rows = 0;
    for( size_t k = 0; k <= K_; k++ ) rows += Y_[k + 1];
    vRows_.resize( rows );
    vOrders_.resize( K_ + 1 );
    size_t r = 0;
    for( size_t k = 0; k <= K_; k++ ){
        vOrders_[k] = vRows_.data() + r;
        for( size_t y = 0; y < Y_[k + 1]; y++ ) vRows_[r++] = v_.data() + off_[k] + y * W_;
    }
    sRows_.resize( Y_[K_ + 1] );
    for( size_t y = 0; y < Y_[K_ + 1]; y++ ) sRows_[y] = s_.data() + y * W_;
    aRows_.resize( K_ + 1 );
    for( size_t k = 0; k <= K_; k++ ) aRows_[k] = a_.data() + k * W_;
}

Motif::Motif( size_t length, size_t K, std::vector<float> alpha, float** v_bg, size_t k_bg, float glob_q )
    : W_( length ), K_( K ), q_( glob_q ), v_bg_( v_bg ), k_bg_( k_bg ){
    if( W_ < 1 || W_ > BAMM_MAX_MOTIF_WIDTH ){
        // the device path takes motifs of up to BAMM_MAX_MOTIF_WIDTH columns (include/bamm_b200.h); the reference has no such limit
        std::cerr << "Error: motif width " << W_ << " (including --extend columns) is outside [1, " << BAMM_MAX_MOTIF_WIDTH
                  << "], the range of the B200 path." << std::endl;
        exit( 1 );
    }
    allocate();
    if( v_bg_ == NULL ){
        // uniform order-2 background (reference: src/init/Motif.cpp:19-28)
        k_bg_ = 2;
        size_t total = 0;
        for( size_t k = 0; k <= k_bg_; k++ ) total += Y_[k + 1];
        ownBg_.resize( total );
        ownBgRows_.resize( k_bg_ + 1 );
        size_t o = 0;
        for( size_t k = 0; k <= k_bg_; k++ ){
            ownBgRows_[k] = ownBg_.data() + o;
            for( size_t y = 0; y < Y_[k + 1]; y++ ) ownBg_[o++] = powf( 1.0f / Y_[1], static_cast<float>( k + 1 ) );
        }
        v_bg_ = ownBgRows_.data();
    }
    for( size_t k = 0; k <= K_; k++ ) for( size_t j = 0; j < W_; j++ ) a_[k * W_ + j] = alpha[k];
    bindViews();
}

Motif::Motif( const Motif& o )
    : isInitialized_( true ), C_( o.C_ ), W_( o.W_ ), K_( o.K_ ), q_( o.q_ ), v_bg_( o.v_bg_ ), k_bg_( o.k_bg_ ),
      ownBg_( o.ownBg_ ), Y_( o.Y_ ), off_( o.off_ ), v_( o.v_ ), p_( o.p_ ), a_( o.a_ ), s_( o.s_ ), n_( o.n_ ){
    if( !ownBg_.empty() ){
        ownBgRows_.resize( k_bg_ + 1 );
        size_t off = 0;
        for( size_t k = 0; k <= k_bg_; k++ ){ ownBgRows_[k] = ownBg_.data() + off; off += Y_[k + 1]; }
        v_bg_ = ownBgRows_.data();
    }
    bindViews();
}

Motif::~Motif(){}

// reference: Motif::initFromBindingSites, src/init/Motif.cpp:134-189. One site per line; flanks are filled with
// random bases drawn with libc util::rand31() (same expression, so the stream stays aligned with the reference).
void Motif::initFromBindingSites( char* indir, size_t l_flank, size_t r_flank ){
    std::ifstream file( indir );
    std::string site;
    while( std::getline( file, site ).good() ){
        C_++;
        for( size_t i = 0; i < l_flank; i++ )
            site.insert( site.begin(), Alphabet::getBase( static_cast<uint8_t>( static_cast<uint8_t>( util::rand31() ) % static_cast<uint8_t>( Y_[1] ) + 1 ) ) );
        for( size_t i = 0; i < r_flank; i++ )
            site.insert( site.end(), Alphabet::getBase( static_cast<uint8_t>( static_cast<uint8_t>( util::rand31() ) % static_cast<uint8_t>( Y_[1] ) + 1 ) ) );
        if( site.length() != W_ ){
            fprintf( stderr, "Error: Length of binding site on line %d differs.\nBinding sites should have the same length.\n", ( int )C_ );
            exit( 1 );
        }
        if( site.length() < K_ + 1 ){
            fprintf( stderr, "Error: Length of binding site sequence is shorter than model order.\n" );
            exit( 1 );
        }
        for( size_t k = 0; k <= K_; k++ ){
            for( size_t j = k; j < W_; j++ ){
                size_t y = 0;
                for( size_t a = 0; a <= k; a++ ) y += Y_[a] * ( static_cast<size_t>( Alphabet::getCode( site[j - a] ) ) - 1 );
                n_[off_[k] + y * W_ + j]++;
            }
        }
    }
    calculateV( n_ );
    calculateP();
    isInitialized_ = true;
}

// reference: Motif::calculateV, src/init/Motif.cpp:403-428
void Motif::calculateV( const std::vector<int>& n ){
    for( size_t y = 0; y < Y_[1]; y++ ){
        for( size_t j = 0; j < W_; j++ ){
            v_[y * W_ + j] = ( n[y * W_ + j] + a_[j] * v_bg_[0][y] ) / ( static_cast<float>( C_ ) + a_[j] );
        }
    }
    for( size_t k = 1; k <= K_; k++ ){
        float* vk = v_.data() + off_[k];
        const float* vk1 = v_.data() + off_[k - 1];
        const int* nk = n.data() + off_[k];
        const int* nk1 = n.data() + off_[k - 1];
        const float* ak = a_.data() + k * W_;
        for( size_t y = 0; y < Y_[k + 1]; y++ ){
            const size_t y2 = y % Y_[k], yk = y / Y_[1];
            for( size_t j = 0; j < k; j++ ) vk[y * W_ + j] = vk1[y2 * W_ + j];
            for( size_t j = k; j < W_; j++ ){
                vk[y * W_ + j] = ( nk[y * W_ + j] + ak[j] * vk1[y2 * W_ + j] ) / ( nk1[yk * W_ + j - 1] + ak[j] );
            }
        }
    }
}

// reference: Motif::initFromPWM, src/init/Motif.cpp:192-333. Order 0 comes from the PWM; higher orders are counted
// from one site per sequence, sampled from the PWM's posterior with a default-seeded std::mt19937 and
// std::discrete_distribution (libstdc++, like the reference). The reference runs the sampling loop under OpenMP with
// a shared generator (a race); here it is serial, which equals the reference's 1-thread behaviour.
void Motif::initFromPWM( float** PWM, size_t asize, SequenceSet* posSeqset, float q ){
    q_ = q;
    std::fill( n_.begin(), n_.end(), 0 );
    for( size_t j = 0; j < W_; j++ ){
        float norm = 0.0f;
        for( size_t y = 0; y < asize; y++ ){
            v_[y * W_ + j] = ( PWM[y][j] <= 1.e-8 ) ? 1.e-8 : PWM[y][j];
            norm += v_[y * W_ + j];
        }
        for( size_t y = 0; y < asize; y++ ) v_[y * W_ + j] /= norm;
    }
    std::vector<float> score( asize * W_ );
    for( size_t y = 0; y < asize; y++ ) for( size_t j = 0; j < W_; j++ ) score[y * W_ + j] = v_[y * W_ + j] / v_bg_[0][y];

    std::vector<Sequence*> posSet = posSeqset->getSequences();
    std::mt19937 rngx;
    size_t count = 0;
    std::vector<Sequence*> kept;
    for( Sequence* s : posSet ){ if( s->getL() < W_ ) count++; else kept.push_back( s ); }
    if( count > 0 ) std::cout << "Note: " << count << " short sequences have been neglected for sampling PWM." << std::endl;

    // Large sets: the posteriors, the draws and the counting run on the device (bamm_seqset_sample_pwm_sites); the host
    // only advances the generator the way std::discrete_distribution would (one generate_canonical<double,53> per
    // sequence, in order). BAMM_DEVICE_PWMINIT=1 / 0 forces either path.
    const char* force = getenv( "BAMM_DEVICE_PWMINIT" );
    if( !kept.empty() && ( force ? atoi( force ) != 0 : kept.size() >= 20000 ) ){
        std::vector<double> uniforms( kept.size() );
        for( size_t n = 0; n < kept.size(); n++ ) uniforms[n] = std::generate_canonical<double, std::numeric_limits<double>::digits>( rngx );
        std::vector<uint64_t> indices;
        bool whole = false;
        SequenceSet* set = SequenceSet::commonSet( kept, indices, &whole );
        static_assert( sizeof( int ) == sizeof( int32_t ), "count table type" );
        BAMM_CHECK( bamm_seqset_sample_pwm_sites( set->device(), whole ? NULL : indices.data(), indices.size(), static_cast<int>( W_ ),
                                                  static_cast<int>( K_ ), static_cast<int>( asize ), score.data(), q, uniforms.data(),
                                                  reinterpret_cast<int32_t*>( n_.data() ), NULL ) );
        kept.clear();                                            // nothing left for the host loop
    }
    for( size_t n = 0; n < kept.size(); n++ ){
        const size_t LW1 = kept[n]->getL() - W_ + 1;
        size_t* kmer = kept[n]->getKmer();
        std::vector<float> r( LW1 + 1 );
        float normFactor = 0.0f;
        const float pos0 = 1.0f - q;
        const float pos1 = q / static_cast<float>( LW1 );
        for( size_t i = 1; i <= LW1; i++ ){
            r[i] = 1.0f;
            for( size_t j = 0; j < W_; j++ ) r[i] *= score[( kmer[i - 1 + j] % asize ) * W_ + j];
            r[i] *= pos1;
            normFactor += r[i];
        }
        r[0] = pos0;
        normFactor += r[0];
        for( size_t i = 0; i <= LW1; i++ ) r[i] /= normFactor;
        std::discrete_distribution<size_t> posterior( r.begin(), r.end() );
        const size_t z = posterior( rngx );
        if( z > 0 ){
            for( size_t k = 0; k <= K_; k++ ){
                for( size_t j = 0; j < W_; j++ ) n_[off_[k] + ( kmer[z - 1 + j] % Y_[k + 1] ) * W_ + j]++;
            }
        }
    }
    for( size_t k = 1; k <= K_; k++ ){
        float* vk = v_.data() + off_[k];
        const float* vk1 = v_.data() + off_[k - 1];
        const int* nk = n_.data() + off_[k];
        const int* nk1 = n_.data() + off_[k - 1];
        const float* ak = a_.data() + k * W_;
        for( size_t y = 0; y < Y_[k + 1]; y++ ){
            const size_t y2 = y % Y_[k], yk = y / Y_[1];
            for( size_t j = 0; j < k; j++ ) vk[y * W_ + j] = vk1[y2 * W_ + j];
            for( size_t j = k; j < W_; j++ ){
                vk[y * W_ + j] = ( nk[y * W_ + j] + ak[j] * vk1[y2 * W_ + j] ) / ( nk1[yk * W_ + j - 1] + ak[j] );
            }
        }
    }
    calculateP();
    isInitialized_ = true;
}

// reference: Motif::initFromBaMM, src/init/Motif.cpp:336-397 (.ihbcp layout: per position K+1 lines, then a blank line)
void Motif::initFromBaMM( char* indir, size_t l_flank, size_t r_flank ){
    std::ifstream file( indir, std::ifstream::in );
    if( !file.is_open() ){
        std::cerr << "Error: Input BaMM file cannot be opened!" << std::endl;
        exit( 1 );
    }
    const float uniform = 1.0f / static_cast<float>( Y_[1] );
    auto fillColumn = [&]( size_t j ){
        for( size_t k = 0; k <= K_; k++ ) for( size_t y = 0; y < Y_[k + 1]; y++ ) v_[off_[k] + y * W_ + j] = uniform;
    };
    for( size_t j = 0; j < l_flank; j++ ) fillColumn( j );
    std::string line;
    for( size_t j = l_flank; j < W_ - r_flank; j++ ){
        for( size_t k = 0; k <= K_; k++ ){
            std::getline( file, line );
            std::stringstream number( line );
            for( size_t y = 0; y < Y_[k + 1]; y++ ) number >> v_[off_[k] + y * W_ + j];
        }
        std::getline( file, line );
    }
    for( size_t j = W_ - r_flank; j < W_; j++ ) fillColumn( j );
    calculateP();
    isInitialized_ = true;
}

// reference: Motif::updateV, src/init/Motif.h:95-136 (host version for callers that hold counts in reference layout;
// the EM wrapper runs the same arithmetic on the device, k_update_model)
void Motif::updateV( float*** n, float** alpha, size_t K ){
    assert( isInitialized_ );
    std::vector<float> sumN( W_, 0.f );
    for( size_t y = 0; y < Y_[1]; y++ ) for( size_t j = 0; j < W_; j++ ) sumN[j] += n[0][y][j];
    for( size_t y = 0; y < Y_[1]; y++ ){
        for( size_t j = 0; j < W_; j++ ){
            v_[y * W_ + j] = ( n[0][y][j] + alpha[0][j] * v_bg_[0][y] ) / ( sumN[j] + alpha[0][j] );
        }
    }
    for( size_t k = 1; k < K + 1; k++ ){
        float* vk = v_.data() + off_[k];
        const float* vk1 = v_.data() + off_[k - 1];
        for( size_t y = 0; y < Y_[k + 1]; y++ ){
            const size_t y2 = y % Y_[k], yk = y / Y_[1];
            for( size_t j = 0; j < k; j++ ) vk[y * W_ + j] = vk1[y2 * W_ + j];
            for( size_t j = k; j < W_; j++ ){
                vk[y * W_ + j] = ( n[k][y][j] + alpha[k][j] * vk1[y2 * W_ + j] ) / ( n[k - 1][yk][j - 1] + alpha[k][j] );
            }
        }
    }
}

// reference: Motif::calculateP, src/init/Motif.cpp:430-469
void Motif::calculateP(){
    for( size_t j = 0; j < W_; j++ ) for( size_t y = 0; y < Y_[1]; y++ ) p_[y * W_ + j] = v_[y * W_ + j];
    for( size_t k = 1; k <= K_; k++ ){
        for( size_t y = 0; y < Y_[k + 1]; y++ ){
            const size_t yk = y / Y_[1];
            float* pk = p_.data() + off_[k] + y * W_;
            for( size_t j = 0; j < k; j++ ){
                // positions whose context reaches left of the motif: motif factors for the part inside, background outside
                float prod = 1;
                for( size_t i = 0; i <= j; i++ ) prod *= v_[off_[k - i] + ( y / Y_[i] ) * W_ + ( j - i )];
                for( size_t i = j + 1; i <= k; i++ ){
                    if( ( k - i ) <= k_bg_ || k <= k_bg_ ) prod *= v_bg_[k - i][y / Y_[i]];
                    else                                    prod *= v_bg_[k_bg_][y / Y_[1] % Y_[k_bg_ + 1]];
                }
                pk[j] = prod;
            }
            for( size_t j = k; j < W_; j++ ) pk[j] = v_[off_[k] + y * W_ + j] * p_[off_[k - 1] + yk * W_ + j - 1];
        }
    }
}

// reference: Motif::calculateLogS, src/init/Motif.cpp:471-483
void Motif::calculateLogS( float** Vbg, size_t K_bg ){
    const float* vK = v_.data() + off_[K_];
    for( size_t y = 0; y < Y_[K_ + 1]; y++ ){
        const size_t y_bg = y % Y_[K_bg + 1];
        for( size_t j = 0; j < W_; j++ ) s_[y * W_ + j] = logf( vK[y * W_ + j] + 1e-5f ) - logf( Vbg[K_bg][y_bg] );
    }
}

// reference: Motif::calculateLinearS, src/init/Motif.cpp:485-494
void Motif::calculateLinearS( float** Vbg, size_t K_bg ){
    const float* vK = v_.data() + off_[K_];
    for( size_t y = 0; y < Y_[K_ + 1]; y++ ){
        const size_t y_bg = y % Y_[K_bg + 1];
        for( size_t j = 0; j < W_; j++ ) s_[y * W_ + j] = vK[y * W_ + j] / Vbg[K_bg][y_bg];
    }
}

void Motif::print(){
    for( size_t j = 0; j < W_; j++ ){
        for( size_t k = 0; k <= K_; k++ ){
            float sum = 0.f;
            for( size_t y = 0; y < Y_[k + 1]; y++ ){
                std::cout << std::scientific << v_[off_[k] + y * W_ + j] << '\t';
                sum += v_[off_[k] + y * W_ + j];
            }
            std::cout << "\t sum = " << sum << std::endl;
        }
        std::cout << std::endl;
    }
}

// .ihbcp (conditional probabilities) and .ihbp (probabilities): per motif position one line per order, 3 significant
// digits in scientific notation, blank line between positions (reference: src/init/Motif.cpp:515-547)
void Motif::write( char* odir, std::string basename ){
    const std::string stem = std::string( odir ) + '/' + basename;
    std::ofstream fv( ( stem + ".ihbcp" ).c_str() );
    std::ofstream fp( ( stem + ".ihbp" ).c_str() );
    for( size_t j = 0; j < W_; j++ ){
        for( size_t k = 0; k <= K_; k++ ){
            for( size_t y = 0; y < Y_[k + 1]; y++ ){
                fv << std::scientific << std::setprecision( 3 ) << v_[off_[k] + y * W_ + j] << ' ';
                fp << std::scientific << std::setprecision( 3 ) << p_[off_[k] + y * W_ + j] << ' ';
            }
            fv << std::endl;
            fp << std::endl;
        }
        fv << std::endl;
        fp << std::endl;
    }
}
