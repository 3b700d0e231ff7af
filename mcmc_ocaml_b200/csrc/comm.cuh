// comm.cuh -- what the other translation units use from comm.cu: the communicator's context, the device collectives
// and the one exchange by which every rank-pooled entry point reports a failure on any rank.
#pragma once
#include <vector>

#include "common.cuh"

namespace mg {

mg_ctx *mg_comm_ctx(const mg_comm *c);

// NCCL on the context's stream; one rank: nothing to do (a copy when d_send != d_recv)
int comm_broadcast_dev(mg_comm *c, void *d_buf, size_t nbytes, int root);
int comm_allgather_dev(mg_comm *c, const void *d_send, void *d_recv, size_t nbytes_per_rank);

// All-gather one fixed-size host record per rank, with the rank's status in front.  Every rank enters the collective
// whatever its rc is (rec is not read when rc != MG_OK, but nbytes must be the same on every rank).  Returns, in this
// order: rc, when this rank had failed (its own message stays); the collective's own error; the status of the lowest
// failing rank r, with the message "<what>: rank r failed"; otherwise MG_OK, with all = the records in rank order.
int comm_gather(mg_comm *c, int rc, const void *rec, size_t nbytes, std::vector<uint8_t> &all, const char *what);

template <class T>
int comm_gather(mg_comm *c, int rc, const std::vector<T> &rec, std::vector<T> &all, const char *what) {
  std::vector<uint8_t> b;
  if ((rc = comm_gather(c, rc, rec.data(), sizeof(T) * rec.size(), b, what))) return rc;
  all.resize(b.size() / sizeof(T));
  memcpy(all.data(), b.data(), b.size());
  return MG_OK;
}

}  // namespace mg
