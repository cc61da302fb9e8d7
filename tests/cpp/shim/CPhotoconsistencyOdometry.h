// TEST INFRASTRUCTURE.  Stand-in for the reference's phovo/include/CPhotoconsistencyOdometry.h and the
// Matrix.h typedefs it uses, so that the drop-in adapter (include/CPhotoconsistencyOdometryCuda.h) and
// tests/cpp/frame_alignment_app.cpp compile without a checkout of the original project.  It declares
// what the adapter derives from and nothing else: the matrix types as thin subclasses of Eigen::Matrix
// (Matrix.h:44-483) and the abstract solver with its seven pure virtuals (base :137-179).  cv:: and
// Eigen:: are the stand-ins of oracle/shim.  tests/cpp/build_adapter_test.sh uses the reference's own
// header instead when REF names a checkout of the original project.
#ifndef PHOVO_TEST_SHIM_CPHOTOCONSISTENCY_ODOMETRY_H_
#define PHOVO_TEST_SHIM_CPHOTOCONSISTENCY_ODOMETRY_H_

#include "opencv2/imgproc/imgproc.hpp"
#include "Eigen/Core"

namespace phovo
{
namespace Numeric
{
template< class T > class Matrix33RowMajor : public Eigen::Matrix< T, 3, 3, Eigen::RowMajor > {};
template< class T > class Matrix44RowMajor : public Eigen::Matrix< T, 4, 4, Eigen::RowMajor > {};
template< class T > class VectorCol6 : public Eigen::Matrix< T, 6, 1 > {};
template< class T > class VectorCol4 : public Eigen::Matrix< T, 4, 1 > {};
} // namespace Numeric

template< class TPixel, class TCoordinate >
class CPhotoconsistencyOdometry
{
public:
  typedef TPixel                PixelType;
  typedef cv::Mat_< PixelType > IntensityImageType;
  typedef TCoordinate                CoordinateType;
  typedef cv::Mat_< CoordinateType > DepthImageType;
  typedef Numeric::Matrix33RowMajor< CoordinateType > Matrix33Type;
  typedef Numeric::Matrix44RowMajor< CoordinateType > Matrix44Type;
  typedef Numeric::VectorCol6< CoordinateType >       Vector6Type;
  typedef Numeric::VectorCol4< CoordinateType >       Vector4Type;

  virtual ~CPhotoconsistencyOdometry() {}
  virtual void SetIntrinsicMatrix( const Matrix33Type & intrinsicMatrix ) = 0;
  virtual void SetSourceFrame( const IntensityImageType & intensityImage, const DepthImageType & depthImage ) = 0;
  virtual void SetTargetFrame( const IntensityImageType & intensityImage, const DepthImageType & depthImage ) = 0;
  virtual void SetInitialStateVector( const Vector6Type & initialStateVector ) = 0;
  virtual void Optimize() = 0;
  virtual Vector6Type GetOptimalStateVector() const = 0;
  virtual Matrix44Type GetOptimalRigidTransformationMatrix() const = 0;
};
} // namespace phovo

#endif
