// k_pointset.cu -- explicit kernel instantiations (see launch.cuh): point sets
#include "launch.cuh"
INSTANTIATE_SMP(SlotPointset<true>)
INSTANTIATE_SMP(SlotPointset<false>)
