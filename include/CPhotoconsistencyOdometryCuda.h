/*
 * CPhotoconsistencyOdometryCuda.h -- drop-in C++ adapter: the reference's solver interface on top of
 * the B200 C ABI (phovo_b200.h).
 *
 * It derives from the reference's own abstract class
 *   phovo::CPhotoconsistencyOdometry<TPixel,TCoordinate>      (phovo/include/CPhotoconsistencyOdometry.h:137-179)
 * and has the same non-virtual extras as the analytic solver it replaces
 *   ReadConfigurationFile / SetMinDepth / SetMaxDepth           (CPhotoconsistencyOdometryAnalytic.h:448-457, 581-607)
 * so both apps switch to it by adding one `#elif USE_PHOTOCONSISTENCY_ODOMETRY_METHOD == 3` branch
 * (INTEGRATION.md).  The header only touches `.rows .cols .data .step` of the cv::Mat_ arguments and
 * `operator()` of the Eigen-derived matrix types, and it includes "CPhotoconsistencyOdometry.h" by
 * name: that is the reference's own header.  tests/cpp/build_adapter_test.sh compiles against it,
 * unmodified, when REF names a checkout of the original project, and otherwise against the stand-in
 * tests/cpp/shim/CPhotoconsistencyOdometry.h; OpenCV and Eigen are the stand-ins of oracle/shim.
 *
 * Error behaviour: the reference returns void and never checks anything; this adapter keeps the
 * void signatures and throws std::runtime_error when the C ABI reports a failure (bad call order,
 * CUDA error, unreadable config, non-finite result) -- a crash-loud superset of the reference's
 * silence.  Nothing is thrown across the C ABI itself.  There is no CPU path: constructing the
 * object on a machine without a CUDA device throws.
 */
#ifndef _CPHOTOCONSISTENCY_ODOMETRY_CUDA_
#define _CPHOTOCONSISTENCY_ODOMETRY_CUDA_

#include <stdexcept>
#include <string>
#include <vector>

#include "CPhotoconsistencyOdometry.h"
#include "phovo_b200.h"

namespace phovo
{
namespace Cuda
{

namespace detail
{
template< class T > struct DepthTypeOf;
template<> struct DepthTypeOf< double > { enum { value = PHOVO_DEPTH_F64 }; };
template<> struct DepthTypeOf< float >  { enum { value = PHOVO_DEPTH_F32 }; };
} // namespace detail

/*!B200 implementation of the photoconsistency alignment behind the reference interface.
 * TPixel must be an 8-bit type (the apps use unsigned char), TCoordinate double or float.*/
template< class TPixel, class TCoordinate >
class CPhotoconsistencyOdometryCuda :
    public CPhotoconsistencyOdometry< TPixel, TCoordinate >
{
public:
  typedef CPhotoconsistencyOdometry< TPixel, TCoordinate > Superclass;

  typedef typename Superclass::CoordinateType     CoordinateType;
  typedef typename Superclass::IntensityImageType IntensityImageType;
  typedef typename Superclass::DepthImageType     DepthImageType;
  typedef typename Superclass::Matrix33Type       Matrix33Type;
  typedef typename Superclass::Matrix44Type       Matrix44Type;
  typedef typename Superclass::Vector6Type        Vector6Type;

  /*!mode: PHOVO_MODE_ANALYTIC_REF reproduces CPhotoconsistencyOdometryAnalytic bit-for-bit in
   * semantics (including AN:253); PHOVO_MODE_ANALYTIC_FIXED uses the Maxima-exact Jacobian;
   * PHOVO_MODE_CERES evaluates the CPhotoconsistencyOdometryCeres residual; PHOVO_MODE_BIOBJECTIVE is
   * CPhotoconsistencyOdometryBiObjective (photometric + depth rows).*/
  explicit CPhotoconsistencyOdometryCuda( int device = 0, int mode = PHOVO_MODE_ANALYTIC_REF ) : m_Ctx( 0 )
  {
    static_assert( sizeof( TPixel ) == 1, "intensity images must be 8-bit" );
    if( phovo_create( device, &m_Ctx ) != PHOVO_OK )
      throw std::runtime_error( std::string( "phovo_create: " ) + phovo_last_error( 0 ) );
    Check( phovo_set_mode( m_Ctx, mode ), "phovo_set_mode" );
  }

  ~CPhotoconsistencyOdometryCuda() { phovo_destroy( m_Ctx ); }

  /*!Sets the minimum depth distance (m) to consider a certain pixel valid (AN:448-451).*/
  void SetMinDepth( const CoordinateType minD )
  {
    phovo_config cfg; Check( phovo_get_config( m_Ctx, &cfg ), "phovo_get_config" );
    Check( phovo_set_depth_range( m_Ctx, double( minD ), cfg.max_depth ), "phovo_set_depth_range" );
  }

  /*!Sets the maximum depth distance (m) to consider a certain pixel valid (AN:454-457).*/
  void SetMaxDepth( const CoordinateType maxD )
  {
    phovo_config cfg; Check( phovo_get_config( m_Ctx, &cfg ), "phovo_get_config" );
    Check( phovo_set_depth_range( m_Ctx, cfg.min_depth, double( maxD ) ), "phovo_set_depth_range" );
  }

  /*!Sets the 3x3 intrinsic pinhole matrix (AN:460-463).*/
  void SetIntrinsicMatrix( const Matrix33Type & intrinsicMatrix )
  {
    double K[9];
    for( int i = 0; i < 3; i++ )
      for( int j = 0; j < 3; j++ )
        K[ 3 * i + j ] = double( intrinsicMatrix( i, j ) );
    Check( phovo_set_intrinsics( m_Ctx, K ), "phovo_set_intrinsics" );
  }

  /*!Sets the source (Intensity+Depth) frame (AN:466-476). Depth in meters.*/
  void SetSourceFrame( const IntensityImageType & intensityImage,
                       const DepthImageType & depthImage )
  {
    if( intensityImage.rows != depthImage.rows || intensityImage.cols != depthImage.cols )
      throw std::runtime_error( "SetSourceFrame: intensity and depth image sizes differ" );
    Check( phovo_set_source( m_Ctx, reinterpret_cast< const uint8_t * >( intensityImage.data ), size_t( intensityImage.step ),
                             depthImage.data, detail::DepthTypeOf< TCoordinate >::value, size_t( depthImage.step ), 1.0,
                             intensityImage.rows, intensityImage.cols ), "phovo_set_source" );
  }

  /*!Sets the target (Intensity+Depth) frame (AN:479-491). The analytic and Ceres solvers ignore the
   * depth image like the reference does; the photometric + depth solver (PHOVO_MODE_BIOBJECTIVE,
   * CPhotoconsistencyOdometryBiObjective.h:567-579) uses it.*/
  void SetTargetFrame( const IntensityImageType & intensityImage,
                       const DepthImageType & depthImage )
  {
    Check( phovo_set_target( m_Ctx, reinterpret_cast< const uint8_t * >( intensityImage.data ), size_t( intensityImage.step ),
                             intensityImage.rows, intensityImage.cols ), "phovo_set_target" );
    phovo_config cfg; Check( phovo_get_config( m_Ctx, &cfg ), "phovo_get_config" );
    if( cfg.mode == PHOVO_MODE_BIOBJECTIVE )
      Check( phovo_set_target_depth( m_Ctx, depthImage.data, detail::DepthTypeOf< TCoordinate >::value,
                                     size_t( depthImage.step ), 1.0 ), "phovo_set_target_depth" );
  }

  /*!Initializes the state vector to a certain value (AN:494-497): x, y, z, yaw, pitch, roll.*/
  void SetInitialStateVector( const Vector6Type & initialStateVector )
  {
    double s[6];
    for( int i = 0; i < 6; i++ ) s[i] = double( initialStateVector( i ) );
    Check( phovo_set_initial_state( m_Ctx, s ), "phovo_set_initial_state" );
  }

  /*!Launches the least-squares optimization process (AN:500-563). Blocking.*/
  void Optimize()
  {
    Check( phovo_optimize( m_Ctx ), "phovo_optimize" );
  }

  /*!Returns the optimal state vector (AN:566-569).*/
  Vector6Type GetOptimalStateVector() const
  {
    double s[6];
    Check( phovo_get_state( m_Ctx, s ), "phovo_get_state" );
    Vector6Type v;
    for( int i = 0; i < 6; i++ ) v( i ) = CoordinateType( s[i] );
    return v;
  }

  /*!Returns the optimal 4x4 rigid transformation matrix (AN:572-578, eigenPose).*/
  Matrix44Type GetOptimalRigidTransformationMatrix() const
  {
    double rt[16];
    Check( phovo_get_rt( m_Ctx, rt ), "phovo_get_rt" );
    Matrix44Type Rt;
    for( int i = 0; i < 4; i++ )
      for( int j = 0; j < 4; j++ )
        Rt( i, j ) = CoordinateType( rt[ 4 * i + j ] );
    return Rt;
  }

  /*!Reads the configuration parameters from a .yml file (AN:581-607 / CE:526-576).*/
  void ReadConfigurationFile( const std::string & fileName )
  {
    Check( phovo_load_config_yaml( m_Ctx, fileName.c_str() ), "phovo_load_config_yaml" );
  }

  // ---- extensions (not in the reference) ---------------------------------------------------
  /*!VO loop (PhotoconsistencyVisualOdometry.cpp:222-223,256-257): the previous target frame becomes
   * the source frame without rebuilding its intensity pyramid; only its depth is uploaded.*/
  void PromoteTargetToSource( const DepthImageType & depthImage )
  {
    Check( phovo_promote_target_to_source( m_Ctx, depthImage.data, detail::DepthTypeOf< TCoordinate >::value,
                                           size_t( depthImage.step ), 1.0 ), "phovo_promote_target_to_source" );
  }

  /*!phovo::warpImage (CPhotoconsistencyOdometry.h:73-134) on the GPU: same arguments as the
   * reference's free function; the apps call it after Optimize() to display the alignment.*/
  void WarpImage( const IntensityImageType & intensityImage, const DepthImageType & depthImage,
                  IntensityImageType & warpedIntensityImage, const Matrix44Type & Rt,
                  const Matrix33Type & intrinsicMatrix, const int level = 0 )
  {
    double rt[16], K[9];
    for( int i = 0; i < 4; i++ ) for( int j = 0; j < 4; j++ ) rt[ 4 * i + j ] = double( Rt( i, j ) );
    for( int i = 0; i < 3; i++ ) for( int j = 0; j < 3; j++ ) K[ 3 * i + j ] = double( intrinsicMatrix( i, j ) );
    warpedIntensityImage.create( intensityImage.rows, intensityImage.cols );
    Check( phovo_warp_image( m_Ctx, reinterpret_cast< const uint8_t * >( intensityImage.data ), size_t( intensityImage.step ),
                             depthImage.data, detail::DepthTypeOf< TCoordinate >::value, size_t( depthImage.step ), 1.0,
                             intensityImage.rows, intensityImage.cols, rt, K, level,
                             reinterpret_cast< uint8_t * >( warpedIntensityImage.data ), size_t( warpedIntensityImage.step ),
                             0, 0, 0, 0 ), "phovo_warp_image" );
  }

  /*!Executed Gauss-Newton iterations of the last Optimize() with their normal equations.*/
  std::vector< phovo_iter_stats > GetIterationStats() const
  {
    std::vector< phovo_iter_stats > out( size_t( phovo_num_iter_stats( m_Ctx ) ) );
    for( size_t i = 0; i < out.size(); i++ ) Check( phovo_get_iter_stats( m_Ctx, int( i ), &out[i] ), "phovo_get_iter_stats" );
    return out;
  }

  /*!Device time (ms, CUDA events) of the last frame setup and of the last Optimize().*/
  void GetTimings( float & setupMs, float & optimizeMs ) const
  {
    Check( phovo_get_timings( m_Ctx, &setupMs, &optimizeMs ), "phovo_get_timings" );
  }

  phovo_ctx * GetContext() { return m_Ctx; }

private:
  CPhotoconsistencyOdometryCuda( const CPhotoconsistencyOdometryCuda & );
  CPhotoconsistencyOdometryCuda & operator=( const CPhotoconsistencyOdometryCuda & );

  void Check( int rc, const char * what ) const
  {
    if( rc != PHOVO_OK )
      throw std::runtime_error( std::string( what ) + ": " + phovo_last_error( m_Ctx ) );
  }

  phovo_ctx * m_Ctx;
};

} //end namespace Cuda
} //end namespace phovo

#endif
