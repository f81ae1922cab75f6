// kh/record_line.hpp -- one kmer_pair record as a line of the reference's k-mer file.  The single definition of that
// format: the GPU formatter (kc_lines_kernel, via count_core.cuh) and host C++ code (kh::pair_lines in kmer_counter.hpp)
// both call kc_record_to_line, so the two can never disagree.
#pragma once

#ifdef __CUDACC__
#define KH_RECORD_LINE_FN __host__ __device__ __forceinline__
#else
#define KH_RECORD_LINE_FN inline
#endif

namespace kh {

// a kmer_pair record as a line of the reference's k-mer file (read_kmers.hpp:64-76 parses exactly this): K bases, a
// blank, the backward and the forward extension letter, '\n' -- K + 4 bytes
KH_RECORD_LINE_FN void kc_record_to_line(const unsigned char* rec, int k, unsigned char* line) {
    const int pl = (k + 3) >> 2;
    for (int i = 0; i < k; ++i)                                             // packing.hpp:94-107 (unpackKmer)
        line[i] = (unsigned char)(0x54474341u >> (8u * ((unsigned)(rec[i >> 2] >> (6 - 2 * (i & 3))) & 3u)));   // "ACGT"
    line[k] = ' ';
    line[k + 1] = rec[pl];
    line[k + 2] = rec[pl + 1];
    line[k + 3] = '\n';
}

}  // namespace kh
