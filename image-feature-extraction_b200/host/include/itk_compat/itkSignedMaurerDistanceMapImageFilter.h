// itk::SignedMaurerDistanceMapImageFilter (ife/Filters/SignedMaurerDistanceMapImageFilter.h).
#ifndef IFE_B200_ITK_COMPAT_SIGNED_MAURER_DISTANCE_MAP_IMAGE_FILTER_H
#define IFE_B200_ITK_COMPAT_SIGNED_MAURER_DISTANCE_MAP_IMAGE_FILTER_H
#include "itkImage.h"
#include "ife/Filters/SignedMaurerDistanceMapImageFilter.h"

namespace itk {
using ife::SignedMaurerDistanceMapImageFilter;
}
#endif
