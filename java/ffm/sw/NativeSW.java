package sw ;

import java.lang.foreign.Arena ;
import java.lang.foreign.FunctionDescriptor ;
import java.lang.foreign.Linker ;
import java.lang.foreign.MemorySegment ;
import java.lang.foreign.SymbolLookup ;
import java.lang.invoke.MethodHandle ;
import java.nio.charset.StandardCharsets ;

import static java.lang.foreign.ValueLayout.ADDRESS ;
import static java.lang.foreign.ValueLayout.JAVA_BYTE ;
import static java.lang.foreign.ValueLayout.JAVA_INT ;
import static java.lang.foreign.ValueLayout.JAVA_LONG ;

/**
 * Panama FFM (JDK 22+) binding of libswb200.so -- the C ABI declared in include/swb200.h.
 * NOT COMPILED OR RUN in the build environment (no JDK there); it shows the exact binding a
 * maintainer adds.  One process-wide context on CUDA device 0 (or -Dswb.device=N).
 *
 * Errors: every native call returns 0 or a negative code; this class turns a non-zero
 * code into an unchecked RuntimeException carrying swb_last_error(), because
 * Function3.call declares no checked exception (reference SmithWaterman.java:62).
 */
final class NativeSW
{
	static final Linker LINKER = Linker.nativeLinker() ;
	static final Arena ARENA = Arena.global() ;
	static final SymbolLookup LIB = SymbolLookup.libraryLookup(
			System.getProperty( "swb.library" , "libswb200.so" ) , ARENA ) ;

	static MethodHandle h( String name , FunctionDescriptor fd )
	{
		return LINKER.downcallHandle( LIB.find(name).orElseThrow() , fd ) ;
	}

	static final MethodHandle LAST_ERROR  = h( "swb_last_error" , FunctionDescriptor.of(ADDRESS) ) ;
	static final MethodHandle CREATE      = h( "swb_create" , FunctionDescriptor.of(JAVA_INT, JAVA_INT, JAVA_LONG, ADDRESS) ) ;
	static final MethodHandle REFSET_LOAD = h( "swb_refset_load" , FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle REFSET_FREE = h( "swb_refset_free" , FunctionDescriptor.ofVoid(ADDRESS) ) ;
	static final MethodHandle ALIGN       = h( "swb_align" , FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle ALIGN_PAIR  = h( "swb_align_pair" , FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle ALIGN_HITS  = h( "swb_align_hits" , FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle RESULT_FREE = h( "swb_result_free" , FunctionDescriptor.ofVoid(ADDRESS) ) ;
	static final MethodHandle RESULT_HITS = h( "swb_result_hits" , FunctionDescriptor.of(ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle MULTI_ALIGN_HITS = h( "swb_multi_align_hits" , FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle MULTI_RESULT_HITS = h( "swb_multi_result_hits" , FunctionDescriptor.of(ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle ALIGN_ALL_HITS = h( "swb_align_all_hits" , FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle RESULT_HIT_OFFSETS = h( "swb_result_hit_offsets" , FunctionDescriptor.of(ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle RESULT_HIT_LIST = h( "swb_result_hit_list" , FunctionDescriptor.of(ADDRESS, ADDRESS) ) ;
	static final MethodHandle MULTI_ALIGN_ALL_HITS = h( "swb_multi_align_all_hits" , FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS) ) ;
	static final MethodHandle MULTI_RESULT_HIT_OFFSETS = h( "swb_multi_result_hit_offsets" , FunctionDescriptor.of(ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle MULTI_RESULT_HIT_LIST = h( "swb_multi_result_hit_list" , FunctionDescriptor.of(ADDRESS, ADDRESS) ) ;
	static final MethodHandle SCORES      = h( "swb_result_scores" , FunctionDescriptor.of(ADDRESS, ADDRESS) ) ;
	static final MethodHandle REF_TOTALS  = h( "swb_result_ref_totals" , FunctionDescriptor.of(ADDRESS, ADDRESS) ) ;
	static final MethodHandle CELL_OFFS   = h( "swb_result_cell_offsets" , FunctionDescriptor.of(ADDRESS, ADDRESS) ) ;
	static final MethodHandle CELL_COUNT  = h( "swb_result_pair_cell_count" , FunctionDescriptor.of(JAVA_LONG, ADDRESS, JAVA_LONG) ) ;
	static final MethodHandle PAIR_CELL   = h( "swb_result_pair_cell" , FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, ADDRESS) ) ;
	static final MethodHandle MATERIALIZE = h( "swb_result_materialize" , FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG) ) ;

	/** swb_align flags (swb200.h); F_BOTH_STRANDS: every read and its reverse complement, o = 2r + strand */
	static final int F_SCORES_ONLY = 1 , F_NO_FETCH = 2 , F_TIE_GT = 4 , F_BOTH_STRANDS = 8 ;

	/** process-wide engine context (thread-safe on the native side) */
	static final MemorySegment CTX = create() ;

	private static MemorySegment create()
	{
		try( Arena a = Arena.ofConfined() )
		{
			MemorySegment out = a.allocate( ADDRESS ) ;
			check( (int) CREATE.invokeExact( Integer.getInteger("swb.device",0).intValue() , 0L , out ) ) ;
			return out.get( ADDRESS , 0 ) ;
		}
		catch( RuntimeException e ) { throw e ; }
		catch( Throwable t ) { throw new RuntimeException( t ) ; }
	}

	static void check( int rc )
	{
		if( rc == 0 ) return ;
		String msg ;
		try { msg = ((MemorySegment) LAST_ERROR.invokeExact()).reinterpret(4096).getString(0) ; }
		catch( Throwable t ) { msg = "?" ; }
		throw new RuntimeException( "libswb200 error " + rc + ": " + msg ) ;
	}

	/** sequences -> (concatenated Latin-1 bytes, int64 offsets[n+1]) in native memory */
	static MemorySegment[] pack( Arena a , java.util.List<String> seqs )
	{
		long total = 0 ;
		for( String s : seqs ) total += s.length() ;
		MemorySegment bytes = a.allocate( Math.max(total,1) ) ;
		MemorySegment offs = a.allocate( JAVA_LONG , seqs.size() + 1L ) ;
		long p = 0 ;
		for( int k = 0 ; k < seqs.size() ; k++ )
		{
			offs.setAtIndex( JAVA_LONG , k , p ) ;
			byte[] b = seqs.get(k).getBytes( StandardCharsets.ISO_8859_1 ) ;
			MemorySegment.copy( b , 0 , bytes , JAVA_BYTE , p , b.length ) ;
			p += b.length ;
		}
		offs.setAtIndex( JAVA_LONG , seqs.size() , p ) ;
		return new MemorySegment[]{ bytes , offs } ;
	}
}
