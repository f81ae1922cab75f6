# Build without Python: the CUDA library, the reference's CLI per K, the generator.  Same flags as
# cs267_hw3_b200/build.py and tools/kmergen.py (those are what __graft_entry__.build() and the tests use).
#
#   make                 libkh_b200.so + kmer_hash_19 kmer_hash_31 kmer_hash_51 + kmer_count + tools/gen_kmers
#   make KS="21 27"      other k-mer lengths (2..61)
#   make check           CPU test suite;  make check-gpu  the GPU parity suite (needs a B200)
NVCC      ?= nvcc
CXX       ?= g++
NVCCFLAGS ?= -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17
CXXFLAGS  ?= -O2 -std=c++17 -pthread
KS        ?= 19 31 51

PKG  := cs267_hw3_b200
LIB  := $(PKG)/libkh_b200.so
CSRC := $(wildcard $(PKG)/csrc/*.cu $(PKG)/csrc/*.cuh)
HDRS := $(wildcard include/*.h include/*.hpp include/kh/*.hpp)
CLIS := $(addprefix kmer_hash_,$(KS))

all: $(LIB) $(CLIS) kmer_count tools/gen_kmers tools/libkmergen.so

$(LIB): $(CSRC) include/kh_capi.h include/kh/record_line.hpp
	$(NVCC) $(NVCCFLAGS) -Xcompiler -fPIC -shared $(PKG)/csrc/capi.cu $(PKG)/csrc/count.cu -o $@

kmer_hash_%: src/kmer_hash.cpp $(HDRS) $(LIB)
	$(CXX) $(CXXFLAGS) -DKMER_LEN=$* -Iinclude $< -L$(PKG) -lkh_b200 -Wl,-rpath,$(abspath $(PKG)) -o $@

kmer_count: src/kmer_count.cpp include/kh_capi.h include/kh/kmer_counter.hpp include/kh/sharded_counter.hpp include/kh/sharded_host.hpp include/kh/record_line.hpp $(LIB)
	$(CXX) $(CXXFLAGS) -Iinclude $< -L$(PKG) -lkh_b200 -Wl,-rpath,$(abspath $(PKG)) -o $@

tools/gen_kmers: tools/kmer_gen.cpp
	$(CXX) $(CXXFLAGS) -DKG_MAIN $< -o $@

tools/libkmergen.so: tools/kmer_gen.cpp
	$(CXX) $(CXXFLAGS) -fPIC -shared $< -o $@

check:
	python -m pytest tests -q -m "not gpu"

check-gpu:
	python -m pytest tests -q -m gpu

clean:
	rm -f $(LIB) $(CLIS) kmer_count tools/gen_kmers tools/libkmergen.so

.PHONY: all check check-gpu clean
