// K6 with mask coefficients (yre_dfl_decode_score_masks): the NM = 32 instantiations of k_decode.cu's kernel, in a
// translation unit of their own so that the detection instantiations compile exactly as before (see k_decode.cu).
#define YRE_DECODE_MASKS
#include "k_decode.cu"
