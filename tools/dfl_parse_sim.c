// dfl_parse_sim.c — CPU model of the LZ77 parse of k_deflate_chunks (otezip_b200/csrc/k_deflate.cuh, phase 1), used to
// choose the match-search scheme of round 2 without spending GPU time: 65,280-byte chunks, 32 positions per step whose
// candidates are read before the step's own insertions, 4-byte hash, greedy parse with lazy evaluation; the size estimate
// is the entropy of the token histograms + extra bits + a header guess (within 1 % of what the GPU encoder produces).
//   gcc -O2 -o dfl_parse_sim tools/dfl_parse_sim.c -lm
//   ./dfl_parse_sim corpus.bin [hb=<hash bits>] [ways=<bucket ways>] [one] [lazy2=1] [twopass=1] [first4] [insall] [rep]
//                   [chain=<depth>] [adapt=<pairs>] [nice=<len>] [best [minm=3|4]]
//   (corpus.bin: 32 x 256 KiB slices of synth.TextPool(seed=5), the corpus of bench.py --workload c5)
// Results that shaped the kernel (ratio on that corpus; zlib level 6: 9.38):
//   hb=12 ways=1 one                      6.85   round 1 (measured on the GPU: 6.87)
//   hb=12 ways=1 one lazy2=1              7.09   + two-step lazy rule            -> compression level 1 (GPU: 7.10)
//   hb=13 / hb=14 ways=1 insall           6.89 / 6.90   more hash bits, all positions inserted: nothing
//   hb=9 ways=8 one                       8.18   eight ways in the same 8 KiB of shared memory
//   hb=9 ways=8 one lazy2=1               8.49   searched at every position      (GPU: 8.52 at 18.9 GB/s)
//   hb=9 ways=8 one lazy2=1 twopass=1     8.23   searched at the token starts of a first pass -> default level (GPU: 8.25 at 29.8 GB/s)
//   hb=9 ways=8 one lazy2=1 twopass=1 adapt=32   8.00   at most 32 (token, way) pairs per step
//   hb=9 ways=8 one lazy2=1 first4        7.05   first way whose four bytes match, no second pass
//   hb=8 ways=16 one / hb=15 chain=16     8.37 / 8.92   (chain=: the ways, then the chain behind the oldest one, to <depth> links)
// Best level (`best`: exact chains over all positions, every position searched on its own, zlib's lazy parse; zlib-6 on
// whole entries 9.38, zlib-9 on independent 65,280-byte chunks 9.69):
//   best hb=15 minm=4 chain=4096 nice=258            9.71   zlib's level-9 search, one-step lazy rule
//   best hb=15 minm=3 chain=4096 nice=258            9.65   minimum match 3 (with TOO_FAR) loses in one Huffman block
//   best hb=15 minm=4 chain=128 nice=128             9.62
//   best hb=14 minm=4 lazy2=1 nice=258 chain=8 / 16 / 32 / 64   8.94 / 9.29 / 9.54 / 9.74   two-step lazy rule
//   best hb=14 minm=4 lazy2=1 nice=258 chain=128     9.91   -> best level (k_deflate_best.cuh)
//   best hb=14 minm=4 lazy2=1 nice=258 chain=256 / 4096   10.00 / 10.01
//   best hb=14 minm=3 lazy2=1 chain=32 9.33; hb=13 = hb=14; nice=128 = nice=258 at chain=64
// A cost-based parse was not modelled: the lazy rule clears the bar with 5 % to spare.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <stdint.h>
#define CHUNK 65280
#define MINM 4
#define MAXM 258
static int ADAPT=0; static int TWOPASS=0, FIRST4=0, NICE=9999; static long npairs_tot=0, nsteps=0; static int HB=12, INSALL=0, REP=0, WAYS=1, MINM3=0, LAZY2=0, CHAIN=0, ONE=0;
static uint32_t rd32(const uint8_t*p){uint32_t v;memcpy(&v,p,4);return v;}
static int mlen_at(const uint8_t*d,uint32_t n,uint32_t p,uint32_t c){uint32_t maxl=n-p<MAXM?n-p:MAXM;uint32_t l=0;while(l<maxl&&d[c+l]==d[p+l])l++;return l;}
static int lsym(int len){ // returns symbol idx 0..28 and extra bits
  static const int base[29]={3,4,5,6,7,8,9,10,11,13,15,17,19,23,27,31,35,43,51,59,67,83,99,115,131,163,195,227,258};
  int s=28; while(base[s]>len)s--; return s;}
static const int lext[29]={0,0,0,0,0,0,0,0,1,1,1,1,2,2,2,2,3,3,3,3,4,4,4,4,5,5,5,5,0};
static int dsym(int dist){static const int base[30]={1,2,3,4,5,7,9,13,17,25,33,49,65,97,129,193,257,385,513,769,1025,1537,2049,3073,4097,6145,8193,12289,16385,24577};int s=29;while(base[s]>dist)s--;return s;}
static const int dext[30]={0,0,0,0,1,1,2,2,3,3,4,4,5,5,6,6,7,7,8,8,9,9,10,10,11,11,12,12,13,13};
static double chunk_bits(const uint8_t*d,uint32_t n){
  uint32_t hs=1u<<HB; uint16_t*ht=calloc(hs*WAYS,2); uint16_t *prev = CHAIN? calloc(65536,2):NULL;
  double hl[286]={0},hd[30]={0}; double xbits=0; uint32_t cur=0; uint32_t lastd=0; long ntok=0;
  uint32_t mlen[64],mdist[64];
  while(cur<n){
    // lookup phase for 32 positions (candidates read before inserts of this step)
    uint32_t cand[32][32]; uint32_t hh[32]; int can[32];
    for(int l=0;l<32;l++){uint32_t p=cur+l;can[l]=p+MINM<=n; if(can[l]){hh[l]=(rd32(d+p)*2654435761u)>>(32-HB); for(int w=0;w<WAYS;w++)cand[l][w]=ht[hh[l]*WAYS+w];}}
    for(int l=0;l<32;l++) if(can[l]){uint32_t p=cur+l; // insert (later lanes override = most recent)
        if(ONE){int later=0; for(int m=l+1;m<32;m++) if(can[m]&&hh[m]==hh[l])later=1; if(later)continue;}
        if(CHAIN) prev[p]=ht[hh[l]*WAYS];
        for(int w=WAYS-1;w>0;w--)ht[hh[l]*WAYS+w]=ht[hh[l]*WAYS+w-1]; ht[hh[l]*WAYS]=p+1;}
    for(int l=0;l<32;l++){mlen[l]=0;mdist[l]=0; if(!can[l])continue; uint32_t p=cur+l;
      int wmax = TWOPASS ? 1 : WAYS;
      if(FIRST4){ for(int w=0;w<WAYS;w++){uint32_t c=cand[l][w]; if(c&&p-(c-1)<=32768&&rd32(d+c-1)==rd32(d+p)){int L=mlen_at(d,n,p,c-1); if(L>=MINM){mlen[l]=L;mdist[l]=p-(c-1);} break;}} continue; }
      for(int w=0;w<wmax;w++){uint32_t c=cand[l][w]; if(c&&p-(c-1)<=32768){int L=mlen_at(d,n,p,c-1); if(L>=MINM&&L>(int)mlen[l]){mlen[l]=L;mdist[l]=p-(c-1);}}}
      if(CHAIN){uint32_t c=cand[l][WAYS-1]; for(int k=0;k<CHAIN&&c;k++){c=prev[c-1]; if(!c||p-(c-1)>32768)break; int L=mlen_at(d,n,p,c-1); if(L>=MINM&&L>(int)mlen[l]){mlen[l]=L;mdist[l]=p-(c-1);}}}
    }
    if(TWOPASS){ for(int pass=0;pass<TWOPASS;pass++){ uint32_t i=0; uint32_t lim=n-cur<32?n-cur:32; int start[32]={0};
        while(i<lim){uint32_t L=mlen[i],Ln=(i+1<32)?mlen[i+1]:0; uint32_t Ln2=(i+2<32)?mlen[i+2]:0; start[i]=1; if(L>=MINM&&Ln<=L&&!(LAZY2&&Ln2>L+1)) i+=L; else i++;}
        nsteps++; int t1=0; for(int l=0;l<32;l++) t1+=start[l]; int wlim=WAYS; if(ADAPT){ wlim=1+ADAPT/(t1?t1:1); if(wlim>WAYS)wlim=WAYS; if(wlim<2)wlim=2;} for(int l=0;l<32;l++) if(start[l]&&can[l]&&(int)mlen[l]<NICE){uint32_t p=cur+l; npairs_tot+=wlim-1; for(int w=1;w<wlim;w++){uint32_t c=cand[l][w]; if(c&&p-(c-1)<=32768){int L=mlen_at(d,n,p,c-1); if(L>=MINM&&L>(int)mlen[l]){mlen[l]=L;mdist[l]=p-(c-1);}}}}
    } }
    uint32_t i=0; uint32_t lim=n-cur<32?n-cur:32;
    while(i<lim){uint32_t L=mlen[i],Ln=(i+1<32)?mlen[i+1]:0; 
      uint32_t Ln2=(i+2<32)?mlen[i+2]:0; if(L>=MINM&&Ln<=L&&!(LAZY2&&Ln2>L+1)&&!(LAZY2==2&&L<6&&mdist[i]>4096)){int s=lsym(L);hl[257+s]++;xbits+=lext[s];int ds=dsym(mdist[i]);hd[ds]++;xbits+=dext[ds];lastd=mdist[i];
         if(INSALL){ // insert positions beyond the window covered by this match
           for(uint32_t q=cur+32;q<cur+i+L&&q+MINM<=n;q++){uint32_t h=(rd32(d+q)*2654435761u)>>(32-HB); if(CHAIN)prev[q]=ht[h*WAYS]; for(int w=WAYS-1;w>0;w--)ht[h*WAYS+w]=ht[h*WAYS+w-1]; ht[h*WAYS]=q+1;}}
         i+=L;}
      else{hl[d[cur+i]]++;i++;}
      ntok++;}
    cur+=i;
  }
  hl[256]=1; double tl=0,td=0,bits=0; for(int i=0;i<286;i++)tl+=hl[i]; for(int i=0;i<30;i++)td+=hd[i];
  for(int i=0;i<286;i++)if(hl[i])bits+=-hl[i]*log2(hl[i]/tl); for(int i=0;i<30;i++)if(hd[i])bits+=-hd[i]*log2(hd[i]/td);
  free(ht); if(prev)free(prev); return bits*1.005+xbits+ 90*8 + 5*8; }
// BEST: the scheme of k_deflate_best (k_deflate_best.cuh).  Hash chains over every position of the chunk (hash of the first
// MINB bytes, HB bits; chains are exact: the warp-serial insertion of the kernel links equal-hash lanes in position order),
// every position searched on its own to CHAIN links with an early exit at NICE (longest wins, the nearer on equal lengths),
// then zlib's lazy parse over the per-position matches (a match is taken unless the next position has a longer one;
// lazy2=1 also looks two ahead), a length-3 match farther than 4,096 bytes is dropped (zlib's TOO_FAR).
static int BEST=0, MINB=4;
static double chunk_bits_best(const uint8_t*d,uint32_t n){
  uint32_t hs=1u<<HB; uint16_t*head=calloc(hs,2); uint16_t*prev=calloc(CHUNK,2); uint16_t*ml=calloc(n+2,2); uint16_t*md=calloc(n+2,2);
  double hl[286]={0},hd[30]={0}; double xbits=0;
  for(uint32_t p=0;p+MINB<=n;p++){uint32_t v=rd32(d+p); if(MINB==3)v&=0xFFFFFF; uint32_t h=(v*2654435761u)>>(32-HB); prev[p]=head[h]; head[h]=p+1;
    uint32_t best=0,bd=0,maxl=n-p<MAXM?n-p:MAXM; uint32_t c=prev[p];
    for(int k=0;k<CHAIN&&c;k++,c=prev[c-1]){ if(p-(c-1)>32768)break; if(d[c-1+best]!=d[p+best])continue; uint32_t L=mlen_at(d,n,p,c-1); if(L>best){best=L;bd=p-(c-1); if(L>=(uint32_t)NICE||L==maxl)break;}}
    if(best>=(uint32_t)MINB&&!(best==3&&bd>4096)){ml[p]=best;md[p]=bd;} }
  uint32_t i=0; while(i<n){uint32_t L=ml[i]; uint32_t Ln=i+1<n?ml[i+1]:0, Ln2=i+2<n?ml[i+2]:0;
    if(L&&Ln<=L&&!(LAZY2&&Ln2>L+1)){int s=lsym(L);hl[257+s]++;xbits+=lext[s];int ds=dsym(md[i]);hd[ds]++;xbits+=dext[ds];i+=L;} else {hl[d[i]]++;i++;}}
  hl[256]=1; double tl=0,td=0,bits=0; for(int k=0;k<286;k++)tl+=hl[k]; for(int k=0;k<30;k++)td+=hd[k];
  for(int k=0;k<286;k++)if(hl[k])bits+=-hl[k]*log2(hl[k]/tl); for(int k=0;k<30;k++)if(hd[k])bits+=-hd[k]*log2(hd[k]/td);
  free(head);free(prev);free(ml);free(md); return bits*1.005+xbits+ 90*8 + 5*8; }
int main(int argc,char**argv){ for(int i=2;i<argc;i++){ if(!strncmp(argv[i],"hb=",3))HB=atoi(argv[i]+3); if(!strcmp(argv[i],"insall"))INSALL=1; if(!strcmp(argv[i],"rep"))REP=1; if(!strncmp(argv[i],"ways=",5))WAYS=atoi(argv[i]+5); if(!strncmp(argv[i],"chain=",6))CHAIN=atoi(argv[i]+6); if(!strcmp(argv[i],"one"))ONE=1; if(!strcmp(argv[i],"best"))BEST=1; if(!strncmp(argv[i],"minm=",5))MINB=atoi(argv[i]+5); if(!strcmp(argv[i],"first4"))FIRST4=1; if(!strncmp(argv[i],"adapt=",6))ADAPT=atoi(argv[i]+6); if(!strncmp(argv[i],"nice=",5))NICE=atoi(argv[i]+5); if(!strncmp(argv[i],"twopass=",8))TWOPASS=atoi(argv[i]+8); if(!strncmp(argv[i],"lazy2=",6))LAZY2=atoi(argv[i]+6);}
  FILE*f=fopen(argv[1],"rb"); fseek(f,0,SEEK_END); long sz=ftell(f); fseek(f,0,SEEK_SET); uint8_t*d=malloc(sz+16); fread(d,1,sz,f); memset(d+sz,0,16);
  double bits=0; for(long e=0;e<sz;e+=262144){long en=sz-e<262144?sz-e:262144; for(long o=0;o<en;o+=CHUNK){uint32_t n=en-o<CHUNK?en-o:CHUNK; bits+=BEST?chunk_bits_best(d+e+o,n):chunk_bits(d+e+o,n);}}
  printf("nice=%d pairs/step %.1f ",NICE,nsteps?(double)npairs_tot/nsteps:0.0); printf("HB=%d ways=%d chain=%d insall=%d rep=%d one=%d ratio %.3f\n",HB,WAYS,CHAIN,INSALL,REP,ONE,sz*8.0/bits); }
