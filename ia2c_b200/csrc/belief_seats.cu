// belief_seats.cu — the frozen-seat (SEATS) instantiations of belief_pairs_episode_kernel (belief.cu) and their launch,
// ia2c::belief_pairs_episode_seats_launch, in a translation unit of their own.  Instantiated next to the other forms of the
// kernel they changed how nvcc compiled those (the SASS of every pre-existing instantiation stays what it was only without
// them), so belief.cu leaves them out and this file compiles the same source with IA2C_BELIEF_SEATS defined.
#define IA2C_BELIEF_SEATS
#include "belief.cu"
