#include <cstdarg>
#include <cstdio>
#include "../../dsp_final_b200/csrc/dspx_internal.cuh"
#include "../../dsp_final_b200/csrc/tables.cuh"
#include "../../dsp_final_b200/csrc/feat_warp8.cuh"
namespace dspx { void set_error(const char*, ...) {} const char* get_error(){return "";} }
using namespace dspx;
int main(){
  for (int P : {512,1024,2048}) for (int nm : {40,64,128}) {
    dspx_plan pl; pl.cfg = dspx_config{44100,P,P/2,0,nm,13,0.0,-1.0,0.97,0,0}; pl.P=P; pl.M=P/2; pl.n_bins=P/2+1;
    build_window(0,P,pl.host.window); build_filterbank(nm,P,44100,0.0,22050.0,pl.host); build_dct2(13,nm,pl.host.dct2);
    std::vector<float> blob; W8Tables tb{}; warp8_build_tables(&pl, blob, tb);
    const int32_t* fd = reinterpret_cast<const int32_t*>(blob.data()+tb.fdesc);
    int mx=0, tot=0; for (int g=0; g<nm; g++){ mx = std::max(mx, fd[4*g+1]); tot += fd[4*g+1]; }
    // count runs / run lengths
    int runs=0, maxrun=0; for (int k=0;k<pl.n_bins;){ int g=pl.host.bin_filt[k]; int e=k; while(e<pl.n_bins && pl.host.bin_filt[e]==g) e++; if (g>=0){runs++; maxrun=std::max(maxrun,e-k);} k=e; }
    printf("P=%d mels=%d rounds=%d n_slots=%d n_segs=%d max_seg_per_filter=%d total=%d runs=%d maxrun=%d tile_floats=%d total_tab=%d\n", P,nm,tb.rounds,tb.n_slots,tb.n_segs,mx,tot,runs,maxrun,tb.tile_floats,tb.total);
  }
}
