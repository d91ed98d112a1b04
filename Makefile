# stereomatching-b200 -- build of the C-ABI library, the host drivers and the oracle.
#
# Keeps the reference Makefile's contract (reference Makefile:4-31): the same binary
# names, `build=debug|timing|release` output directories, -DDEBUG in debug (PPM dumps go
# to par/ and pargh/ for test/diff.sh) and -DNO_WRITES in timing.  What is new: the CUDA
# side is one shared library built for sm_100a, and the drivers are plain C.
#
#   make lib                      stereomatching_b200/libstereo_b200.so
#   make [build=debug]            debug/stereopar debug/stereopar-ghost
#   make build=timing             timing/...
#   make oracle                   oracle/liboracle.so (+ oracle/_ref when /root/reference exists)

build   := debug
CC      := gcc
NVCC    := nvcc
SM_ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := -O3 -std=c++17 $(SM_ARCH) -lineinfo -Xcompiler -fPIC -Xcompiler -Wall
CFLAGS  := -Wall -Wextra -std=gnu11 -Wno-unused-parameter -Iinclude

ifeq ($(build),debug)
    outdir := debug
    CFLAGS += -g -DDEBUG
else ifeq ($(build),timing)
    outdir := timing
    CFLAGS += -O3 -DNO_WRITES
else ifeq ($(build),release)
    outdir := release
    CFLAGS += -O3
else
    $(error error: invalid value for build)
endif

CSRC   := stereomatching_b200/csrc
LIB    := stereomatching_b200/libstereo_b200.so
KOBJS  := $(patsubst %,$(CSRC)/build/%.o,stereo_b200 k_edges k_pack k_direct k_bitslice k_bitslice16 k_bitslice_ru k_bitslice_sub k_bitslice_ru_sub k_step3)

all: lib benchlib $(outdir)/stereopar $(outdir)/stereopar-ghost $(outdir)/stereobatch host/libhostimage.so

lib: $(LIB)

# measurement-only microbenchmarks (INT32 issue peak, host<->device copy peak) for bench.py: its own library,
# nothing of it is in the product
benchlib: benchlib/libsmb_peaks.so

benchlib/libsmb_peaks.so: benchlib/peaks.cu
	$(NVCC) -O3 -std=c++17 $(SM_ARCH) -lineinfo -Xcompiler -fPIC -shared $< -o $@

$(CSRC)/build/%.o: $(CSRC)/%.cu $(CSRC)/sm_common.cuh include/stereo_b200.h
	@mkdir -p $(CSRC)/build
	$(NVCC) $(NVFLAGS) -c $< -o $@

# the five output families of the bit-sliced kernel share its source
$(CSRC)/build/k_bitslice.o $(CSRC)/build/k_bitslice16.o $(CSRC)/build/k_bitslice_ru.o \
    $(CSRC)/build/k_bitslice_sub.o $(CSRC)/build/k_bitslice_ru_sub.o: $(CSRC)/k_bitslice.cuh

$(LIB): $(KOBJS)
	$(NVCC) $(SM_ARCH) -shared $(KOBJS) -o $@

# make dev: the development build (libstereo_b200_dev.so) with the experiment hooks (SMB_* environment
# variables, -DSMB_DEV) compiled in; the shipped library has none of them.  Select it with
# STEREO_B200_LIB=.../libstereo_b200_dev.so (tools/exp_shapes.py).  DEVFLAGS adds further -D switches.
DEVLIB   := stereomatching_b200/libstereo_b200_dev.so
DEVKOBJS := $(patsubst $(CSRC)/build/%,$(CSRC)/build_dev/%,$(KOBJS))
dev: $(DEVLIB)

$(CSRC)/build_dev/%.o: $(CSRC)/%.cu $(CSRC)/sm_common.cuh include/stereo_b200.h
	@mkdir -p $(CSRC)/build_dev
	$(NVCC) $(NVFLAGS) -DSMB_DEV $(DEVFLAGS) -c $< -o $@

$(CSRC)/build_dev/k_bitslice.o $(CSRC)/build_dev/k_bitslice16.o $(CSRC)/build_dev/k_bitslice_ru.o \
    $(CSRC)/build_dev/k_bitslice_sub.o $(CSRC)/build_dev/k_bitslice_ru_sub.o: $(CSRC)/k_bitslice.cuh

$(DEVLIB): $(DEVKOBJS)
	$(NVCC) $(SM_ARCH) -shared $(DEVKOBJS) -o $@

$(outdir):
	mkdir -p $(outdir)

# Host drivers: plain C, the reference's main()/algorithm() flow over the C ABI.
$(outdir)/stereopar: host/driver.c host/hostimage.c host/hostimage.h include/stereo_b200.h $(LIB) | $(outdir)
	$(CC) $(CFLAGS) -DSM_VARIANT=0 host/driver.c host/hostimage.c -o $@ \
	    -Lstereomatching_b200 -lstereo_b200 -Wl,-rpath,'$$ORIGIN/../stereomatching_b200' -lz -lm

$(outdir)/stereopar-ghost: host/driver.c host/hostimage.c host/hostimage.h include/stereo_b200.h $(LIB) | $(outdir)
	$(CC) $(CFLAGS) -DSM_VARIANT=1 host/driver.c host/hostimage.c -o $@ \
	    -Lstereomatching_b200 -lstereo_b200 -Wl,-rpath,'$$ORIGIN/../stereomatching_b200' -lz -lm

# whole pairs over every GPU of the box through the multi-GPU entry of the C ABI (no reference counterpart)
$(outdir)/stereobatch: host/batch.c include/stereo_b200.h $(LIB) | $(outdir)
	$(CC) $(CFLAGS) host/batch.c -o $@ \
	    -Lstereomatching_b200 -lstereo_b200 -Wl,-rpath,'$$ORIGIN/../stereomatching_b200' -lz

# hostimage as a shared object, for the CPU tests of the PNG reader / PPM writer
host/libhostimage.so: host/hostimage.c host/hostimage.h
	$(CC) -Wall -Wextra -std=gnu11 -O2 -fPIC -shared host/hostimage.c -o $@ -lz

oracle:
	$(MAKE) -C oracle liboracle.so
	if [ -d /root/reference/src ]; then $(MAKE) -C oracle ref; fi

clean:
	-rm -rf debug timing release $(CSRC)/build $(CSRC)/build_dev $(LIB) $(DEVLIB) benchlib/libsmb_peaks.so

.PHONY: all lib dev benchlib oracle clean
