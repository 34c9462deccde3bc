// Per-call values of the persistent head kernels (kernels_head2.cu): everything that changes from step to step (batch size and
// pointers, training flag, barrier / mailbox epochs).  The pointers that never change after pamrec_bind travel in Head2 (head2.h).
#pragma once
#include "kernels.h"

namespace pamrec {

struct HeadDyn {
  int B, T, Bg, training, world, rank;
  double cntN, cntB;
  const int* mask; const float* y_sat; const float* y_play; const float* plays;
  float fuzhu_w, order_w; int sm_group;
  unsigned* bar;                                    // [0] arrivals [2] error word [32] release epoch (own 128-byte line)
  uint32_t p2p_epoch; int p2p_slot0; uint32_t* p2p_err;
  uint4* peer_ll[kP2PMaxWorld];                     // flag-in-data mailboxes [slot][rank][kP2PMaxDoubles] (kernels.h:p2p_ll_offset)
  unsigned long long* trace;                        // [32] %globaltimer of the kernel start ([31]) and of every barrier release; may be null
  float* pred;                                      // scoring (row-stationary kernels): sigmoid(logit 0) per row, or null
  unsigned long long* trace_cta;                    // debug: [16 barriers][256 CTAs] %globaltimer of every CTA's arrival; may be null
  int keep_aw;                                      // scoring: also keep the pooling weights in pool.aw (pamrec_attention); 0 elsewhere
};

}  // namespace pamrec
