/* TEST INFRASTRUCTURE -- pieces of apriltag_oracle.c shared with classic_detector.c (same library). */
#ifndef ORACLE_INTERNAL_H_
#define ORACLE_INTERNAL_H_
#include "apriltag_oracle.h"

void orc_i_to_gray(const orc_config *c, const uint8_t *in, uint8_t *gray);
void orc_i_decimate(const uint8_t *gray, int W, int f, uint8_t *out, int w, int h);
void orc_i_gaussian_blur(uint8_t *im, int w, int h, float quad_sigma);
void orc_i_threshold(const uint8_t *im, int w, int h, int min_white_black_diff, uint8_t *minmax_out, uint8_t *out);
int orc_i_min_tag_width(const orc_config *c);
int orc_i_family_slots(const orc_config *c);
const orc_family *orc_i_family(const orc_config *c, int slot);
void orc_i_border_polarities(const orc_config *c, int *normal_border, int *reversed_border);
float orc_i_quad_decode(const orc_config *c, const orc_family *fam, const uint8_t *im, int W, int H, const double *Hm, int *id,
                        int *hamming, int *rotation);
void orc_i_fill_detection(orc_detection *d, int family, int id, int hamming, float margin, int rotation, const double *Hm);
int orc_i_reconcile(orc_detection *d, int n);
void orc_i_h_project(const double *H, double x, double y, double *ox, double *oy);
#endif
