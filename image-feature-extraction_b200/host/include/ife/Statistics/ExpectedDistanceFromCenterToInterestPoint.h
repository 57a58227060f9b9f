// The probability-weighted mean of the signed distance to a structure's contour: after a classifier
// has produced a per-voxel probability map (of emphysema, say), how far from the structure -- in
// millimetres, negative inside it -- that probability sits.  The reference's header of this name
// computes it from itk::SignedMaurerDistanceMapImageFilter; this is this project's signature, on the GPU
// (ife_cuda_expected_signed_distance: the map is never written, and the sum is deterministic).
//   E = sum weight * d / sum weight over the voxels where region != 0 (every voxel without a region),
//   d the signed, non-squared map of center (!= 0), with the image's spacing.
// Throws ExceptionObject (IFE_E_INVALID) for a geometry mismatch, a negative or non-finite weight, a
// zero weight sum or a center without contour voxels.
#ifndef IFE_B200_EXPECTED_DISTANCE_FROM_CENTER_TO_INTEREST_POINT_H
#define IFE_B200_EXPECTED_DISTANCE_FROM_CENTER_TO_INTEREST_POINT_H
#include "ife/Context.h"
#include "ife/Image.h"

namespace ife {

inline double ExpectedDistanceFromCenterToInterestPoint(const Image<unsigned char>& center, const Image<float>& weight,
                                                        const Image<unsigned char>* region = nullptr,
                                                        bool insideIsPositive = false) {
  const Geometry& g = center.GetGeometry();
  if (weight.GetSize() != g.size || (region && region->GetSize() != g.size))
    throw ExceptionObject(IFE_E_INVALID, "ExpectedDistanceFromCenterToInterestPoint: the images' sizes differ");
  double e = 0.0;
  CudaContext& c = CudaContext::Instance();
  c.Check(ife_cuda_expected_signed_distance(c.Handle(), center.GetBufferPointer(), weight.GetBufferPointer(),
                                            region ? region->GetBufferPointer() : nullptr, g.size.data(),
                                            g.spacing.data(), insideIsPositive ? IFE_SDM_INSIDE_POSITIVE : 0, &e,
                                            IFE_MEM_HOST));
  return e;
}

}  // namespace ife
#endif
