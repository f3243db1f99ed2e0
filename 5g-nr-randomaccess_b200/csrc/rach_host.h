/* rach_host.h -- internal host helpers shared by rach_engine.cu and the test emulator. */
#ifndef RACH_HOST_H
#define RACH_HOST_H
#include <stddef.h>
#include "rach_gpu.h"

int ra_host_validate(const ra_params* p, char* err, size_t errLen);
int ra_host_ring(const ra_params* p);                          /* R: power of two > BI + max(A,5) + Wn */
int ra_host_arrcum(const ra_params* p, int* arrCum, int nOcc); /* returns the final activeCheck */

struct RaPointDev;
void ra_host_fill_point(RaPointDev* pt);                       /* derived fields: magic numbers, hshift, layout */
void ra_host_point(const ra_params* p, RaPointDev* pt);        /* the device view of a validated point, arrCum unset */
void ra_host_point_u0(const ra_params* p, RaPointDev* pt);     /* ... of a variant U0 point (G carries nAccessUE) */
int ra_host_cap3(int variant, const RaPointDev* pt);           /* Msg3 calendar entries per ms slot */

#endif
