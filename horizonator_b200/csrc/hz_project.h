// hz_project.h -- the reference's double-precision projection (horizonator-lib.c:1053-1155), one source for the host
// entry points horizonator_x_from_az() / horizonator_project() (hz_api.cpp) and the annotation kernel k_annotate
// (hz_kernels.cu).
//
// Both translation units are compiled without contraction (-fmad=false on the device, -ffp-contract=off on the host),
// so every operator below is one IEEE rounding on either side.  What can differ is atan2(): glibc's and libdevice's are
// both within an ulp of the exact result but not always the same ulp.  round() and sqrt() are exact on both.
#pragma once
#include <cmath>
#include <cuda_runtime.h>      // __host__ / __device__ (empty for the host compiler)

#define HZ_HD __host__ __device__ inline

HZ_HD double hz_unwrap_near_rad_d(double x, double near)
{
    const double d = (x - near) / (2. * M_PI);
    return (d - round(d)) * 2. * M_PI + near;
}

HZ_HD bool hz_x_from_az(double* x, double* az_ndc_per_rad, double az_rad, double az_rad0, double az_rad1, int width)
{
    az_rad1 = hz_unwrap_near_rad_d(az_rad1 - az_rad0, M_PI) + az_rad0;
    const double center = (az_rad0 + az_rad1) / 2.;
    az_rad = hz_unwrap_near_rad_d(az_rad, center);
    const double per_rad = 2.0 / (az_rad1 - az_rad0);
    const double az_ndc  = (az_rad - center) * per_rad;
    if(!(-1. <= az_ndc && az_ndc <= 1.)) return false;
    if(az_ndc_per_rad != nullptr) *az_ndc_per_rad = per_rad;
    *x = (az_ndc + 1.) / 2. * width - 0.5;                               // NDC [-1,1] -> pixel (-0.5, W-0.5)
    return true;
}

HZ_HD bool hz_project(double* x, double* y, double* range,
                      double lat_viewer, double cos_lat_viewer, double lon_viewer, double ele_viewer,
                      double lat, double lon, double ele,
                      double az_rad0, double az_rad1, int width, int height)
{
    const float Rearth = 6371000.0;
    const double dlat = (lat - lat_viewer) * M_PI / 180;
    const double dlon = (lon - lon_viewer) * M_PI / 180;
    const double east  = dlon * Rearth * cos_lat_viewer;
    const double north = dlat * Rearth;
    const double d2 = east * east + north * north;

    double per_rad;
    if(!hz_x_from_az(x, &per_rad, atan2(east, north), az_rad0, az_rad1, width)) return false;

    const double h = ele - ele_viewer;
    *range = sqrt(d2 + h * h);
    const double aspect = (double)width / (double)height;
    const double el_ndc = atan2(h, sqrt(d2)) * aspect * per_rad;
    if(!(-1. <= el_ndc && el_ndc <= 1.)) return false;
    *y = (-el_ndc + 1.) / 2. * height - 0.5;
    return true;
}
