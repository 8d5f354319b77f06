# Builds, in-tree:
#   vanrijn_b200/lib/libvanrijn_cuda.so  -- the sm_100a kernels + C ABI (include/vanrijn_cuda.h)
#   vanrijn_b200/lib/libvanrijn_host.so  -- C++ host mirror of the reference API (include/vanrijn.hpp) + C shim
#   oracle/libvanrijn_oracle.so          -- CPU oracle (test infrastructure only)
# nvcc cross-compiles for sm_100a without a GPU.  -fmad=false: the reference (rustc) never fuses a*b+c.
NVCC ?= nvcc
# the image exports CXX=/opt/gcc/bin/g++ (a wrapper without libgomp.spec); use the PATH compiler
HOSTCXX = g++
NVFLAGS = -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -std=c++17 --extended-lambda \
          -Xcompiler -fPIC -Xcompiler -fvisibility=hidden
LIBDIR ?= vanrijn_b200/lib
EXTRA ?=
CSRC = vanrijn_b200/csrc
CUDA_DEPS = $(CSRC)/vrj_batch.cuh $(CSRC)/vrj_kernels.cuh $(CSRC)/vrj_traverse.cuh $(CSRC)/vrj_device.cuh \
            $(CSRC)/vrj_internal.h $(CSRC)/rgb_basis_tables.inc include/vanrijn_cuda.h
HOST_DEPS = $(CSRC)/host/vanrijn_host.cpp $(CSRC)/host/host_capi.cpp include/vanrijn.hpp include/vanrijn_cuda.h

all: $(LIBDIR)/libvanrijn_cuda.so $(LIBDIR)/libvanrijn_host.so oracle examples tools

# translation units: the C ABI + scene upload; the device BVH builder; and one object per instantiation of the wavefront
# batch (vrj_batch_inst.cu with -DVRJ_INST=0..5), so `make -j` compiles the kernel variants in parallel
OBJDIR ?= build/obj
BATCH_OBJS = $(OBJDIR)/vrj_batch_0.o $(OBJDIR)/vrj_batch_1.o $(OBJDIR)/vrj_batch_2.o $(OBJDIR)/vrj_batch_3.o \
             $(OBJDIR)/vrj_batch_4.o $(OBJDIR)/vrj_batch_5.o
$(OBJDIR)/vanrijn_cuda.o: $(CSRC)/vanrijn_cuda.cu $(CSRC)/vrj_scene_prep.cuh $(CSRC)/vrj_denoise.cuh $(CUDA_DEPS)
	mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXTRA) -c -o $@ $(CSRC)/vanrijn_cuda.cu
$(OBJDIR)/vrj_batch_%.o: $(CSRC)/vrj_batch_inst.cu $(CUDA_DEPS)
	mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXTRA) -DVRJ_INST=$* -c -o $@ $(CSRC)/vrj_batch_inst.cu
$(OBJDIR)/vrj_bvh_build.o: $(CSRC)/vrj_bvh_build.cu $(CSRC)/vrj_internal.h include/vanrijn_cuda.h
	mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXTRA) -c -o $@ $(CSRC)/vrj_bvh_build.cu

$(LIBDIR)/libvanrijn_cuda.so: $(OBJDIR)/vanrijn_cuda.o $(OBJDIR)/vrj_bvh_build.o $(BATCH_OBJS)
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -shared -o $@ $^ -ldl

$(LIBDIR)/libvanrijn_host.so: $(HOST_DEPS) $(LIBDIR)/libvanrijn_cuda.so
	$(HOSTCXX) -O2 -std=c++17 -fPIC -ffp-contract=off -Wall -Wextra -shared -o $@ \
	    $(CSRC)/host/vanrijn_host.cpp $(CSRC)/host/host_capi.cpp -L$(LIBDIR) -lvanrijn_cuda -pthread -Wl,-rpath,'$$ORIGIN'

oracle:
	$(MAKE) -s -C oracle

# build/vanrijn: the reference's harness (src/main.rs) over the host mirror; build/drop_in_example: doc-test + bench scene
examples: build/vanrijn build/drop_in_example build/merge_bench
build/%: examples/%.cpp $(LIBDIR)/libvanrijn_host.so include/vanrijn.hpp
	mkdir -p build
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -o $@ $< -L$(LIBDIR) -lvanrijn_host -lvanrijn_cuda -Wl,-rpath,'$$ORIGIN/../$(LIBDIR)'
build/merge_bench: tools/merge_bench.cpp $(LIBDIR)/libvanrijn_host.so include/vanrijn.hpp
	mkdir -p build
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -o $@ $< -L$(LIBDIR) -lvanrijn_host -lvanrijn_cuda -Wl,-rpath,'$$ORIGIN/../$(LIBDIR)'
build/vanrijn: examples/vanrijn_main.cpp $(LIBDIR)/libvanrijn_host.so include/vanrijn.hpp
	mkdir -p build
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -o $@ $< -L$(LIBDIR) -lvanrijn_host -lvanrijn_cuda -Wl,-rpath,'$$ORIGIN/../$(LIBDIR)'

# microbenchmark behind roofline.k_trace: dependent 64-byte gathers from L2 / HBM (profiles/r02_l2_gather_peak.json)
tools: build/l2_gather_peak
build/l2_gather_peak: tools/l2_gather_peak.cu
	mkdir -p build
	$(NVCC) -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -o $@ $<

clean:
	rm -f $(LIBDIR)/*.so oracle/*.so
	rm -rf $(OBJDIR) build/vanrijn build/drop_in_example

.PHONY: all oracle clean examples tools
